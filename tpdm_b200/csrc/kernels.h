// tpdm_b200 -- launchers of the bandwidth-bound kernels (kernels.cu).  All return 0 / tpdm_status.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tpdm {

typedef __nv_bfloat16 bf16;

int k_cast_bf16(const float* in, bf16* out, long long n, cudaStream_t s);

// Timesteps(256, flip_sin_to_cos=True, downscale_freq_shift=0): out[b] = [cos(t f_i) | sin(t f_i)], f_i = 10000^(-i/128)
int k_timestep_embedding(const float* timestep, int t_stride, float scale, float* out, int Bt, int rep, cudaStream_t s);

// y[b][j] = (addend ? addend[b][j] : 0) + bias[j] + sum_k W[j][k] * act(x[b][k]);  act: 0 identity, 1 SiLU
int k_gemv_f32(const float* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J,
               int K, int act, cudaStream_t s);
int k_gemv_bf16(const bf16* W, const float* bias, const float* x, int ldx, const float* addend, float* y, int ldy, int Bt, int J,
                int K, int act, cudaStream_t s);

// PatchEmbed: conv 2x2/s2 + bias + centre-cropped pos table.  Sample bl is written to x[bl] and, when dup == 2, x[bl+Bl].
int k_patchify(const float* latents, const float* Wp, const float* bias, const float* pos_table, int pos_max, float* x, int Bl,
               int dup, int C, int Hl, int Wl, int D, float* h1_out, bf16* tpm_x, cudaStream_t s);

struct LnSeg {
  const float* x;      // [batch][rows][D] fp32 residual stream
  bf16* out;           // [batch][rows][D]
  const float* shift;  // [batch] rows of the modulation buffer, stride mod_stride
  const float* scale;
  int rows, batch, mod_stride;
  // E4M3 output instead of `out` (every segment of a launch or none): codes [batch][rows][D] and row scales [batch][rows],
  // quantized per token row by the library's one row quantizer (pack_e4m3x4 in common.cuh)
  uint8_t* out8 = nullptr;
  float* out_scale = nullptr;
};
// LayerNorm(eps 1e-6, no affine) * (1 + scale) + shift for up to two streams in one launch
int k_ln_modulate(const LnSeg* segs, int nseg, int D, cudaStream_t s);
// per row r of x fp32 [rows][K] (K % 4 == 0): codes[r] = E4M3 row quantization of x[r], scales[r] = its scale
int k_quantize_fp8_rows(const float* x, int rows, int K, uint8_t* codes, float* scales, cudaStream_t s);

// norm_out for the sampling loop: LN-modulate both CFG halves (bf16 -> xn for proj_out) and write
// h2 = u + guidance*(c - u), scrambled to pixel order, into tpm_x[bl][pix][D:2D];  optional fp32 h2 [2B][N][D]
int k_norm_out(const float* x, bf16* xn, const float* shift, const float* scale, int mod_stride, int B, int cfg_pairs, int N,
               int D, int g, float guidance, bf16* tpm_x, float* h2_out, cudaStream_t s);

// in-place RMSNorm(eps 1e-6) of the q and k head vectors of tokens [row0, row0+rows) in qkv [Bt][S][3*H*dp]
int k_qk_rmsnorm(bf16* qkv, int Bt, int S, int row0, int rows, int H, int dp, int d, const float* wq, const float* wk,
                 cudaStream_t s);

// pout [Bt][N][4*C] -> velocity [B][C][Hl][Wl] (CFG-combined when cfg_pairs), optional Euler update of latents:
//   latents += (sigma_next - sigma) * v ; history (optional) gets the updated latents
int k_unpatchify(const float* pout, int B, int cfg_pairs, float guidance, int C, int Hl, int Wl, float* velocity,
                 float* latents, const float* sigma, const float* sigma_next, int sigma_stride, float* history,
                 cudaStream_t s);

int k_euler(const float* v, const float* sigma_next, const float* sigma, const float* sample, float* prev, int B, long long n,
            cudaStream_t s);

// out[b] = u[b] + guidance * (c[b] - u[b]) for [B][n] halves of in [2B][n]; also copied to out2 when non-null
int k_cfg_combine(const float* in, float* out, float* out2, int B, int n, float guidance, cudaStream_t s);

// ---- TimePredictor pieces ----
int k_nchw_to_nhwc_bf16(const float* x, bf16* out, int B, int C, int g, cudaStream_t s);
int k_gn_stats(const float* y, double* stats, int B, long long n, cudaStream_t s);  // stats[b] = {sum, sumsq}, pre-zeroed
// a = SiLU( ((y - mean) * rstd * gn_w + gn_b) * (1 + scale) + shift ),  emb[b] = [shift(C) | scale(C)]
int k_gn_mod_silu(const float* y, const double* stats, const float* gn_w, const float* gn_b, const float* emb, float* a, int B,
                  int npix, int C, cudaStream_t s);
int k_conv3x3_s2(const float* a, const float* w, const float* bias, float* y, int B, int g, int C, cudaStream_t s);
// adaptive_avg_pool2d(16,16) -> global max -> fc1 -> SiLU -> fc2 -> exp + eps
int k_tpm_tail(const float* y2, int B, int go, int C, const float* fc1_w, const float* fc1_b, const float* fc2_w,
               const float* fc2_b, float eps, float* alpha_beta, cudaStream_t s);

struct ScheduleArgs {
  const float* alpha_beta;  // [B][2] raw TimePredictor outputs (param1, param2)
  float* sigma_hist;        // [B][T+1]
  float *alphas, *betas, *logprobs;  // [B][T]
  int* masks;               // [B][T]
  int* all_done;            // [T]
  const float* ratios;      // [B][T] injected Beta draws, or null: draw on the device (Philox, Marsaglia-Tsang)
  unsigned long long seed;
  int B, T, step, predict, relative, prediction_type;
  float min_sigma, epsilon;
};
// y[i] = bias[i % C] + sum_s part[s * n + i]: adds up the partial products of a split-K GEMM (n % 4 == 0, C % 4 == 0)
int k_sum_partials(const float* part, int splits, long long n, const float* bias, int C, float* y, cudaStream_t s);
int k_schedule(const ScheduleArgs& a, cudaStream_t s);
// start of a trajectory: sigma_hist[b] = (1, 0, ..., 0), masks = 0, all_done = 0
int k_sample_init(float* sigma_hist, int* masks, int* all_done, int B, int T, cudaStream_t s);

// ---- device-side prompt queue (continuous batching over a fixed number of in-flight slots) ---------------------------
struct QueueArgs {
  const float* alpha_beta;   // [B][2] TimePredictor outputs of this step
  float* sigma_cur;          // [B] sigma the step was run at; advanced / reset in queue_advance
  float* sigma_next;         // [B] written by queue_schedule, consumed by the Euler step
  int* slot_prompt;          // [B] prompt id in flight, -1 = idle
  int* slot_step;            // [B] steps done on that prompt
  int* slot_flush;           // [B] out: prompt id whose final latent must be written out (-1: none)
  int* slot_load;            // [B] out: 1 = a new prompt was assigned to the slot (its inputs must be loaded)
  int* slot_active;          // [B] out: 1 = the slot holds a prompt (set_batch_mask of the next step)
  int* ticket;               // next prompt id; may live in peer / pinned memory shared by several GPUs
  int* out_steps;            // [P]
  float* out_sigmas;         // [P][max_steps + 1] or null
  int* active;               // [1] slots that hold a prompt after this step
  int* idle_flag;            // [1] 1 when active == 0 (skip flag of the next, speculatively enqueued step)
  const int* order;          // [n_prompts] ticket -> prompt id (longest-expected-first scheduling), or null: ticket == prompt id
  const float* init_sigma;   // [P] sigma a prompt enters the queue with (after `init_step` probe steps), or null: 1
  int init_step;             // denoising steps every prompt has already made when it enters the queue (0 without a probe)
  int B, n_prompts, max_steps, relative, prediction_type, init;
  float min_sigma, epsilon;
  // sampled rollouts (predict == 0): ratios_all [P][max_steps] or null (Philox draws from `seed`); records [P][max_steps], each optional
  int predict;
  unsigned long long seed;
  const float* ratios_all;
  float *rec_alphas, *rec_betas, *rec_logprobs;
  // stream mode (tpdm_stream_*): prompt ids are ring entry ids; `order` is the ring [capacity] ticket -> entry, `counters` the
  // stream's kStream* counters and `done_log` [capacity] the completion log.  `ticket`, `n_prompts`, `init_*` are unused.
  int* counters;
  int* done_log;
  int capacity;
};
enum StreamCounter { kStreamSubmitted = 0, kStreamClaimed, kStreamCompleted, kStreamExecuted, kStreamCounters };
int k_queue_schedule(const QueueArgs& a, cudaStream_t s);
int k_queue_advance(const QueueArgs& a, cudaStream_t s);
// stream mode: retire finished slots into the completion log, then every slot without a prompt (finished now or idle before)
// claims the next submitted ticket in slot order.  admit = 1: no step ran (after an admission): only idle slots claim.
int k_stream_advance(const QueueArgs& a, int admit, cudaStream_t s);
// order[(submitted + k) % capacity] = entries[k] for k < n, then submitted += n (one thread, stream-ordered)
constexpr int kStreamPublishMax = 64;
struct StreamEntries {
  int id[kStreamPublishMax];
};
int k_stream_publish(int* order, int* counters, int capacity, const StreamEntries& e, int n, cudaStream_t s);
// per occupied slot b at (prompt, step) = (slot_prompt[b], slot_step[b]): tembs_all[prompt][step] = temb_cfg[b] ([D]) and
// tpm_all[prompt][step] = tpm_x[b] (tpm_elems bf16); either destination may be null
int k_queue_record(const int* slot_prompt, const int* slot_step, int B, int max_steps, int D, const float* temb_cfg, float* tembs_all,
                   const bf16* tpm_x, bf16* tpm_all, long long tpm_elems, cudaStream_t s);
// per slot b: flush -> out_latents[flush] = latents[b]; load -> latents[b] = noise_all[prompt], ctx0 / text_part rows b and B + b
// = ctx0_all / text_all [prompt][0 | 1]
int k_queue_move(const int* slot_prompt, const int* slot_flush, const int* slot_load, int B, long long lat, long long ctx, int D,
                 float* latents, const float* noise_all, float* out_latents, float* ctx0, const float* ctx0_all, float* text_part,
                 const float* text_all, cudaStream_t s);

}  // namespace tpdm
