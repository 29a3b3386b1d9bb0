/* tpdm_b200.h -- C ABI of libtpdm_b200.so: the TPDM adaptive denoising hot path on B200 (sm_100a).
 *
 * The reference (jinkyu032/TPDM) is pure Python and has no FFI; its boundary for this path is the Python call surface
 * (SURVEY.md section 8b).  The Python classes in tpdm_b200/ keep that surface and bind the entry points below with
 * ctypes; each entry point names the reference code it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - every call returns int: 0 = ok, <0 = tpdm_status; the message is in tpdm_last_error() (thread-local);
 *   - no C++ exception crosses the boundary; there is NO CPU fallback: without a CUDA device every compute call fails;
 *   - all tensor arguments are DEVICE pointers, fp32 unless stated, contiguous, borrowed for the duration of the call
 *     and ordered on the cudaStream_t passed as `void* stream` (0 = legacy default stream);
 *   - weights are borrowed for the lifetime of the ctx (the caller keeps them alive; packing is described per field);
 *   - no allocation on the hot path: the caller supplies the workspace a plan is bound to;
 *   - a ctx / plan is bound to the current CUDA device at creation and is not thread-safe.
 */
#ifndef TPDM_B200_H_
#define TPDM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPDM_ABI_VERSION 3

typedef enum tpdm_status {
  TPDM_OK = 0,
  TPDM_ERR_ARG = -1,    /* null / inconsistent argument  -> Python raises ValueError   */
  TPDM_ERR_SHAPE = -2,  /* unsupported shape             -> ValueError                 */
  TPDM_ERR_CUDA = -3,   /* CUDA runtime / driver failure -> RuntimeError               */
  TPDM_ERR_STATE = -4,  /* call order (weights not set, plan not begun ...) -> RuntimeError */
  TPDM_ERR_NOMEM = -5   /* workspace too small           -> RuntimeError               */
} tpdm_status;

/* Mirrors CustomSD3Transformer2DModel.__init__ (src/models/stable_diffusion_3/transformer_sd3.py:91-108) plus the
 * TimePredictor / pipeline knobs (src/models/stable_diffusion_3/modeling_sd3_pnt.py:86,129-140,195-198). */
typedef struct tpdm_config {
  int32_t num_layers;
  int32_t num_heads;
  int32_t head_dim;
  int32_t joint_attention_dim; /* 4096 */
  int32_t pooled_projection_dim; /* 2048 */
  int32_t in_channels;  /* 16 */
  int32_t out_channels; /* 16 */
  int32_t patch_size;   /* 2 (only 2 is supported) */
  int32_t pos_embed_max_size;
  int32_t qk_norm;      /* 0 = None, 1 = "rms_norm" */
  int32_t tpm_channels; /* TimePredictor conv_out_channels, 128 */
  int32_t prediction_type; /* 0 = "alpha_beta", 1 = "mode_concentration" */
  int32_t relative;     /* 1 = sigma_next = sigma * ratio, 0 = sigma - ratio */
  float min_sigma;
  float epsilon;        /* ratio clamp, 1e-3 (modeling_sd3_pnt.py:197) */
  float tpm_epsilon;    /* exp(x) + 1.0 (modeling_sd3_pnt.py:95,115) */
  uint64_t dual_attention_mask; /* bit i set = block i is an SD3.5 dual-attention block (attn2 + 9-chunk norm1),
                                   transformer_sd3.py:104-106,138; 0 for SD3.0 */
} tpdm_config;

/* Per JointTransformerBlock weights (diffusers state-dict names in comments; D = num_heads*head_dim, dp = head_dim
 * rounded up to 64 or 128, Dp = num_heads*dp).  bf16 matrices are row-major [out][in] exactly as nn.Linear stores them. */
typedef struct tpdm_block_weights {
  const void* qkv_w;    /* bf16 [3*Dp][D]  rows: attn.to_q | to_k | to_v, each head padded to dp rows (zeros) */
  const float* qkv_b;   /* [3*Dp] */
  const void* cqkv_w;   /* bf16 [3*Dp][D]  attn.add_q_proj | add_k_proj | add_v_proj */
  const float* cqkv_b;
  const void* out_w;    /* bf16 [D][Dp]    attn.to_out.0 (columns of padded head dims are zero) */
  const float* out_b;
  const void* cout_w;   /* bf16 [D][Dp]    attn.to_add_out            (null in the last block) */
  const float* cout_b;
  const void* ff1_w;    /* bf16 [4D][D]    ff.net.0.proj */
  const float* ff1_b;
  const void* ff2_w;    /* bf16 [D][4D]    ff.net.2 */
  const float* ff2_b;
  const void* cff1_w;   /* ff_context.net.0.proj (null in the last block) */
  const float* cff1_b;
  const void* cff2_w;   /* ff_context.net.2 */
  const float* cff2_b;
  const float* norm_q;  /* [dp] attn.norm_q.weight (zero padded), null when qk_norm == 0 */
  const float* norm_k;
  const float* norm_added_q;
  const float* norm_added_k;
  /* dual-attention blocks only (null otherwise): attn2 = self-attention over the image tokens */
  const void* qkv2_w;   /* bf16 [3*Dp][D]  attn2.to_q | to_k | to_v */
  const float* qkv2_b;
  const void* out2_w;   /* bf16 [D][Dp]    attn2.to_out.0 */
  const float* out2_b;
  const float* norm_q2; /* [dp] attn2.norm_q.weight, null when qk_norm == 0 */
  const float* norm_k2;
} tpdm_block_weights;

typedef struct tpdm_weights {
  const float* patch_w;   /* [D][in_channels*4]  pos_embed.proj.weight flattened (c, p, q) */
  const float* patch_b;   /* [D] */
  const float* pos_table; /* [pos_embed_max_size^2][D]  pos_embed.pos_embed */
  const float* t_w1;      /* [D][256]   time_text_embed.timestep_embedder.linear_1 */
  const float* t_b1;
  const float* t_w2;      /* [D][D]     ...linear_2 */
  const float* t_b2;
  const float* p_w1;      /* [D][pooled] time_text_embed.text_embedder.linear_1 */
  const float* p_b1;
  const float* p_w2;      /* [D][D] */
  const float* p_b2;
  const void* ctx_w;      /* bf16 [D][joint_attention_dim]  context_embedder */
  const float* ctx_b;
  const void* adaln_w;    /* bf16 [R][D]: blocks in order, each norm1.linear (6D rows; 9D for a dual-attention block)
                             followed by norm1_context.linear (6D rows; last block 2D rows), then norm_out.linear (2D).
                             R = 12*D*L - 2*D + 3*D*popcount(dual_attention_mask) */
  const float* adaln_b;   /* [R] */
  const void* proj_w;     /* bf16 [4*out_channels][D]  proj_out */
  const float* proj_b;
  const tpdm_block_weights* blocks; /* HOST array [num_layers]; null = no MMDiT (TimePredictor-only ctx) */
  /* TimePredictor (modeling_sd3_pnt.py:85-126) */
  const void* tpm_conv1_w;    /* bf16 [C1][9][2D]  conv1.weight permuted (oc, ky*3+kx, c); null = no TimePredictor */
  const float* tpm_conv1_b;   /* [C1] */
  const float* tpm_lin_w;     /* [2*C1][D]  norm1.linear */
  const float* tpm_lin_b;
  const float* tpm_gn_w;      /* [C1] norm1.norm.weight */
  const float* tpm_gn_b;
  const float* tpm_conv2_w;   /* [9][C1 in][C1 out]  conv2.weight permuted (ky*3+kx, c, oc) */
  const float* tpm_conv2_b;
  const float* tpm_fc1_w;     /* [128][C1] */
  const float* tpm_fc1_b;
  const float* tpm_fc2_w;     /* [2][128] */
  const float* tpm_fc2_b;
} tpdm_weights;

typedef struct tpdm_ctx tpdm_ctx;
typedef struct tpdm_plan tpdm_plan;

const char* tpdm_last_error(void);
int tpdm_abi_version(void);

int tpdm_create(const tpdm_config* cfg, tpdm_ctx** out);
int tpdm_destroy(tpdm_ctx* ctx);
/* Borrow the packed weights (copied struct, borrowed pointers).  Replaces module construction / load_state_dict
 * (modeling_sd3_pnt.py:144-157, gradio_sd3_inference.py:20-21). */
int tpdm_set_weights(tpdm_ctx* ctx, const tpdm_weights* w);

/* Opt-in FP8 (E4M3) mode of the MMDiT's QKV and FF1 projections.  Per block (host array [num_layers]): E4M3 codes
 * [N][K] of the bf16 matrices of the same name in tpdm_block_weights, quantized per output channel by tpdm_quantize_fp8_rows,
 * and their fp32 scales [N]; cff1_w / cff1_s are null in the last block.  Borrowed for the lifetime of the ctx. */
typedef struct tpdm_fp8_block_weights {
  const void* qkv_w;    /* E4M3 [3*Dp][D] */
  const float* qkv_s;   /* [3*Dp] */
  const void* cqkv_w;   /* E4M3 [3*Dp][D] */
  const float* cqkv_s;
  const void* ff1_w;    /* E4M3 [4D][D] */
  const float* ff1_s;
  const void* cff1_w;   /* E4M3 [4D][D] (null in the last block) */
  const float* cff1_s;
} tpdm_fp8_block_weights;
/* Call after tpdm_set_weights and before the first tpdm_plan_create of the ctx (TPDM_ERR_STATE once a plan has been created).
 * Every plan of the ctx then runs QKV / context QKV and FF1 / context FF1 as E4M3 x E4M3 -> fp32 GEMMs: ln_modulate writes the
 * modulated token rows as E4M3 codes with one scale per row, and the GEMM epilogue applies row scale x channel scale before the
 * bias.  Out-projections, FF2, attention, qk-RMSNorm, SD3.5 attn2, context_embedder, proj_out and the TimePredictor stay bf16.
 * tpdm_plan_workspace_bytes then includes the E4M3 activations and their row scales. */
int tpdm_set_fp8_weights(tpdm_ctx* ctx, const tpdm_fp8_block_weights* blocks);

/* A plan fixes the shapes: `batch` prompts (transformer batch Bt = 2*batch when cfg_pairs != 0, i.e. the loop's
 * cat([latents]*2) at modeling_sd3_pnt.py:524; else Bt = batch), latent side, text tokens, recorded steps. */
size_t tpdm_plan_workspace_bytes(const tpdm_ctx* ctx, int batch, int cfg_pairs, int latent_h, int latent_w, int n_text,
                                 int max_steps);
int tpdm_plan_create(tpdm_ctx* ctx, int batch, int cfg_pairs, int latent_h, int latent_w, int n_text, int max_steps,
                     void* workspace, size_t workspace_bytes, tpdm_plan** out);
int tpdm_plan_destroy(tpdm_plan* plan);

/* CustomSD3Transformer2DModel.forward (transformer_sd3.py:299-409).  Bt rows everywhere.
 *   latents [Bt][C][h][w], timestep [Bt], enc [Bt][T][joint_attention_dim], pooled [Bt][pooled_projection_dim]
 *   -> out_sample [Bt][C][h][w], out_temb [Bt][D], out_h1 [Bt][N][D], out_h2 [Bt][N][D]   (any out may be null) */
int tpdm_mmdit_forward(tpdm_plan* plan, const float* latents, const float* timestep, const float* enc,
                       const float* pooled, float* out_sample, float* out_temb, float* out_h1, float* out_h2,
                       void* stream);

/* TimePredictor.forward (modeling_sd3_pnt.py:100-115) on NCHW input x [Bt][2D][g][g], temb [Bt][D] -> [Bt][2]
 * (Bt = the plan's transformer batch). */
int tpdm_tpm_forward(tpdm_plan* plan, const float* x_nchw, const float* temb, float* out_alpha_beta, void* stream);

/* CustomFlowMatchEulerDiscreteScheduler.custom_step (src/models/model_utilis.py:52-74):
 *   prev = sample + (sigma_next - sigma)[:,None,None,None] * model_output   (fp32; n = elements per sample) */
int tpdm_euler_step(const float* model_output, const float* sigma_next, const float* sigma, const float* sample,
                    float* prev_sample, int batch, long long n, void* stream);

/* The adaptive loop, SD3PredictNextTimeStepModel.forward (modeling_sd3_pnt.py:504-612).
 * begin: latents [batch][C][h][w]; embeddings for the negative and positive prompt [batch][T][J], [batch][pooled].
 *        predict != 0: ratio = Beta(alpha, beta).mode (:567).  predict == 0: ratio = ratios[b][step] when `ratios`
 *        ([batch][max_steps], injected draws) is given, else a device-side Beta(alpha, beta) draw (Philox stream
 *        (seed, sample b, step), Marsaglia-Tsang gammas) standing in for beta_dist.sample() (:569). */
int tpdm_sample_begin(tpdm_plan* plan, const float* latents, const float* neg_embeds, const float* pos_embeds,
                      const float* neg_pooled, const float* pos_pooled, float guidance_scale, int predict,
                      const float* ratios, unsigned long long seed, void* stream);
/* one denoising step `step` (0-based): MMDiT -> CFG -> TPM -> schedule update -> Euler.  No host synchronisation. */
int tpdm_sample_step(tpdm_plan* plan, int step, void* stream);
/* the same step replayed from a CUDA graph: one graph per step index, captured the first time that step runs on this plan and
 * kept while guidance_scale / predict / injected ratios stay as they were (the stream must not be the legacy default stream).
 * Trajectories that draw their ratios on the device (predict == 0 without `ratios`: the seed is a kernel argument) and calls made
 * while tpdm_profile_start is active run the plain step. */
int tpdm_sample_step_graph(tpdm_plan* plan, int step, void* stream);
/* device-resident results; all [batch][max_steps] row-major unless stated */
typedef struct tpdm_sample_state {
  float* latents;        /* [batch][C][h][w] current latents (fp32 master copy) */
  float* velocity;       /* [batch][C][h][w] CFG-combined velocity of the last step */
  float* sigma_hist;     /* [batch][max_steps+1]: column 0 = 1, column k+1 = sigma_next of step k */
  float* alphas;
  float* betas;
  float* logprobs;       /* raw (un-masked) log-prob */
  int32_t* prob_masks;
  int32_t* all_done;     /* [max_steps]: 1 when every sigma_next < min_sigma after that step (modeling_sd3_pnt.py:608) */
  float* tembs;          /* [max_steps][batch][D] CFG-combined temb per step */
  void* tpm_input;       /* bf16 [batch][g][g][2D] NHWC scrambled TPM input of the last step */
  float* history_latents;/* [max_steps][batch][C][h][w] */
} tpdm_sample_state;
int tpdm_sample_state_get(tpdm_plan* plan, tpdm_sample_state* out);

/* ---- training half: TimePredictor replay with gradients, PPO-clip loss, clip + AdamW ----------------------------------
 * Replaces only_predict_logprobs (modeling_sd3_pnt.py:670-726), the ratio / PPO-clip loss / backward of
 * src/train/rloo_trainer.py:485-501 and clip_grad_norm_ + optimizer.step (:505-523) for the TimePredictor (the MMDiT is
 * frozen).  Parameters live in ONE flat fp32 buffer; tpdm_tpm_param_offsets fills 13 element offsets (last = total):
 * conv1.weight as [C1][9][2D] (oc, ky*3+kx, c) | conv1.bias | norm1.linear.weight [2C1][D] | norm1.linear.bias |
 * norm1.norm.weight | norm1.norm.bias | conv2.weight as [9][C1][C1] (tap, c, oc) | conv2.bias | fc1.weight | fc1.bias |
 * fc2.weight | fc2.bias.  Gradients use the same layout, so the data-parallel exchange is one all-reduce of one buffer. */
typedef struct tpdm_tpm_trainer tpdm_tpm_trainer;
int tpdm_tpm_param_offsets(int D, int C1, long long* out13);
size_t tpdm_tpm_trainer_workspace_bytes(int D, int C1, int g, int max_samples);
int tpdm_tpm_trainer_create(int D, int C1, int g, int max_samples, float tpm_epsilon, void* workspace, size_t bytes,
                            tpdm_tpm_trainer** out);
int tpdm_tpm_trainer_destroy(tpdm_tpm_trainer* t);
/* params / grads: flat fp32 device buffers (layout above); conv1_w_bf16: bf16 copy of the first C1*9*2D parameters */
int tpdm_tpm_trainer_bind(tpdm_tpm_trainer* t, float* params, float* grads, void* conv1_w_bf16);
/* x_nhwc bf16 [ns][g][g][2D] (as recorded by tpdm_sample_state.tpm_input), temb [ns][D] -> alpha_beta [ns][2]; keeps the
 * activations the backward needs (x_nhwc / temb are borrowed until the backward has run) */
int tpdm_tpm_train_forward(tpdm_tpm_trainer* t, const void* x_nhwc, const float* temb, int ns, float* alpha_beta,
                           void* stream);
/* dz [ns][2] = d loss / d (fc2 output, i.e. log(alpha - eps), log(beta - eps)); OVERWRITES the bound grads buffer */
int tpdm_tpm_train_backward(tpdm_tpm_trainer* t, const float* dz, void* stream);
/* alpha_beta [mb*T][2] = the TimePredictor outputs in (sample, step) order, sigmas / old_logprobs [mb][T] (old_logprobs with
 * 1.0 at masked steps, as the rollout returns them), advantages [mb] -> new_logprobs [mb][T], dz [mb*T][2] = d loss / d (fc2
 * output), stats4 = {loss, clip fraction, approx KL, mean ratio} (device).  prediction_type as in tpdm_config: with 1 the
 * Beta parameters are alpha = p1 (p2 - 2) + 1, beta = (1 - p1)(p2 - 2) + 1 (modeling_sd3_pnt.py:559-563) and dz carries that
 * chain rule, so the replay scores the same distribution the rollout drew from.  reduce_tail (NULL or 2 floats that sit right
 * behind the flat gradient buffer): {loss or 0 when it is not finite, 1 when it is not finite else 0}; summed by the gradient
 * all-reduce it tells every rank whether ANY rank saw a NaN / Inf loss (rloo_trainer.py:497-500). */
int tpdm_ppo_clip_loss(const float* alpha_beta, const float* sigmas, const float* old_logprobs, const float* advantages,
                       int mb, int T, float min_sigma, float epsilon, int relative, int prediction_type, float cliprange,
                       float tpm_epsilon, float* new_logprobs, float* dz, float* stats4, float* reduce_tail, void* stream);
/* only_predict_logprobs after the TimePredictor (modeling_sd3_pnt.py:699-724): logprobs [mb][T] = Beta log-prob of the
 * recorded ratio (sigma_next / sigma, or sigma - sigma_next when not relative; clamped to [epsilon, 1 - epsilon]), 1.0 where
 * the sample had already finished; dlp_dz [mb*T][2] (may be NULL) = d logprob / d (fc2 output), 0 at finished steps. */
int tpdm_beta_logprob(const float* alpha_beta, const float* sigmas, int mb, int T, float min_sigma, float epsilon,
                      int relative, int prediction_type, float tpm_epsilon, float* logprobs, float* dlp_dz, void* stream);
/* Reward shaping of one RLOO rollout on the device (replaces the Python loops of modeling_sd3_pnt.py:828-841 and :875-901 and
 * the tensor code of rloo_trainer.py:447-461).  alphas / betas / sigmas [batch][steps] fp32 and masks [batch][steps] int32 as
 * the sampler leaves them; last_rewards [batch] (NULL: scores = 0).  Outputs (each may be NULL): kl [batch][steps] =
 * KL(Beta(alpha,beta) || reference) with 0 at masked steps -- the reference is Beta(get_ref_beta(sigma_in, ref_steps)) when
 * `relative`, else Beta(1.4, 11.2); scores [batch] = discounted mean of last_reward (gamma); rlhf_reward = scores -
 * kl_coef * (sum, or mean when mean_kl) of kl; advantages = leave-one-out over the rloo_k repeats (layout: repeats x
 * prompts).  batch <= 1024. */
int tpdm_rollout_shaping(const float* alphas, const float* betas, const float* sigmas, const int* masks,
                         const float* last_rewards, int batch, int steps, int relative, int ref_steps, float gamma,
                         float kl_coef, int mean_kl, int rloo_k, float* kl, float* scores, float* rlhf_reward,
                         float* advantages, void* stream);
/* g = grads * grad_scale; clip to max_grad_norm (<= 0: off); AdamW (decoupled weight decay); a non-finite norm, or
 * *skip_flag != 0 (device float, NULL = none: the all-reduced non-finite-loss count of tpdm_ppo_clip_loss), skips the update
 * (rloo_trainer.py:497-500, 518-520); the first bf16_n parameters are mirrored to bf16_copy.  scratch_sumsq: 1 double on the
 * device (holds |g|^2 after). */
int tpdm_adamw_step(float* params, const float* grads, float* m, float* v, long long n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, float max_grad_norm, int step, float grad_scale, double* scratch_sumsq,
                    void* bf16_copy, long long bf16_n, const float* skip_flag, void* stream);

/* ---- measurement hooks used by bench.py -------------------------------------------------------------------------- */
/* ----------------------------------------------------------------------------------------------------------------
 * Device-side prompt queue (BASELINE config 3: prompts with different trajectory lengths).  The plan's `batch` entries are
 * in-flight SLOTS.  Every prompt runs the same per-prompt trajectory as tpdm_sample_* with batch 1 and predict = 1
 * (modeling_sd3_pnt.py:522-612: the prompt stops at the first sigma_next < min_sigma or at max_steps); a slot whose prompt
 * ended writes its final latent to out_latents[prompt], takes the next ticket (atomicAdd, system scope) and starts on that
 * prompt in the next step -- no host round trip, no collective.  `ticket` is a device-visible int the owner zeroes
 * beforehand; several GPUs of one box share the prompt list by sharing that counter (CUDA IPC / peer memory).
 *   latents_all [P][C][h][w], *_embeds_all [P][T][joint_attention_dim], *_pooled_all [P][pooled_projection_dim]: all P
 *   prompts resident on the device (borrowed until the queue has drained).  Outputs: out_latents [P][C][h][w] (rows of
 *   prompts this plan did not process are left untouched), out_steps [P], out_sigmas [P][max_steps + 1] or NULL.
 * ---------------------------------------------------------------------------------------------------------------- */
size_t tpdm_queue_workspace_bytes(const tpdm_plan* plan, int n_prompts);
/*   Scheduling (all optional): `order` [n_queued] maps ticket t to prompt order[t] (NULL: t), so that a caller can hand out the
 *   prompts longest-expected-first; only the first n_queued tickets exist (<= 0: all n_prompts).  `init_sigma` [P] + `init_step` > 0:
 *   every prompt enters the queue after init_step probe steps made elsewhere -- latents_all then holds the latents AFTER those
 *   steps, init_sigma the sigma they reached, and out_sigmas[prompt][0..init_step] must have been filled by the caller.
 * ---------------------------------------------------------------------------------------------------------------- */
int tpdm_queue_begin(tpdm_plan* plan, int n_prompts, const float* latents_all, const float* neg_embeds_all,
                     const float* pos_embeds_all, const float* neg_pooled_all, const float* pos_pooled_all,
                     float guidance_scale, void* queue_workspace, size_t queue_workspace_bytes, int* ticket,
                     float* out_latents, int* out_steps, float* out_sigmas, const int* order, int n_queued,
                     const float* init_sigma, int init_step, void* stream);
/* Switch a begun queue to sampled rollouts (predict = 0): call after tpdm_queue_begin, before its first tpdm_queue_step.
 * Every prompt then follows the trajectory tpdm_sample_* with predict = 0 gives row `prompt` of one batch of all P prompts.
 * ratios_all [P][max_steps] (NULL: device Beta draws from `seed`, keyed by (prompt, trajectory step) exactly as
 * tpdm_sample_begin keys sample b); records, each [P][max_steps] row-major and each optional: alphas, betas, logprobs (raw),
 * tembs [P][max_steps][D], tpm_inputs bf16 [P][max_steps][g][g][2D].  Entries past a prompt's last step are not written.
 * TPDM_ERR_STATE before tpdm_queue_begin or after one with init_step > 0 (the probe step ran the Beta mode).  A captured
 * queue-step graph is dropped; the seed stays fixed for the drain, so tpdm_queue_step_graph captures the rollout step once. */
int tpdm_queue_set_rollout(tpdm_plan* plan, unsigned long long seed, const float* ratios_all, float* alphas, float* betas,
                           float* logprobs, float* tembs, void* tpm_inputs);
/* one denoising step of every occupied slot, then retire / refill.  No host synchronisation. */
int tpdm_queue_step(tpdm_plan* plan, void* stream);
/* the same step replayed from a CUDA graph captured on the first call (stream must not be the legacy default stream) */
int tpdm_queue_step_graph(tpdm_plan* plan, void* stream);
/* device pointers: *active_slots -> int, slots holding a prompt after the last enqueued step (0 = drained);
 * *slot_prompts -> int[batch] */
int tpdm_queue_status(tpdm_plan* plan, const int** active_slots, const int** slot_prompts);

/* ----------------------------------------------------------------------------------------------------------------
 * Open prompt stream: the device-side prompt queue with admission while it runs (continuous batching for serving).  The
 * plan's `batch` entries are the in-flight slots; prompts live in a ring of `capacity` ENTRIES inside the caller's
 * workspace, each holding the noise latents, the context_embedder output [2][T][D] and pooled-text part [2][D] (uncond, cond),
 * the output latents, step count and sigmas [max_steps + 1] of one request.  The caller owns the free list: an entry is
 * handed to tpdm_stream_submit, and free again once its id was read from the completion log and its outputs were copied.
 * Counters (device int[4]): submitted, claimed, completed, executed steps.  Every stream call and every step is enqueued on
 * ONE stream, so ordering is by stream order; nothing synchronises the host.
 * Steps are tpdm_queue_step / tpdm_queue_step_graph on the plan (one captured graph: the ring, counters, staging and request
 * options never move, so requests with different options never force a recapture).
 * A slot without a prompt -- its trajectory just ended, or it was idle -- takes the next submitted ticket in slot order (no
 * atomics, deterministic); a step of a stream with no active slot is skipped on the device.
 * Each entry also carries its request's options (tpdm_request_options: guidance scale, step cap, predict, seed); a slot that
 * claims the entry runs its CFG combines with that guidance.  A request follows exactly the trajectory tpdm_sample_* gives it
 * with batch 1, guidance_scale, max_steps = its cap and its predict; with predict = 0 the Beta draws are those of
 * tpdm_sample_begin's `seed` = its seed (keyed by (seed, sample 0, step)).  Every executed step records the request's alpha,
 * beta and raw log-prob (tpdm_stream_records).
 * A plan's buffers belong to one driver at a time: the lockstep sampler after tpdm_sample_begin, the closed queue after
 * tpdm_queue_begin, the open stream from tpdm_stream_open to tpdm_stream_close.  Each begin hands the plan to its driver, and a
 * call that needs another owner returns TPDM_ERR_STATE and enqueues nothing:
 *   tpdm_sample_begin, tpdm_queue_begin           refused while a stream is open
 *   tpdm_sample_step, tpdm_sample_step_graph      need the sampler: refused after a later tpdm_queue_begin / tpdm_stream_open
 *   tpdm_queue_set_rollout                        needs the closed queue
 *   tpdm_queue_step, _step_graph, tpdm_queue_status   need the closed queue or the stream: refused after a later
 *                                                 tpdm_sample_begin (its steps would run on the slots the sampler overwrote)
 *   tpdm_stream_open                              refused while a queue owns the plan or a stream is open
 *   tpdm_stream_submit[_options], _status, _records, _close   need the open stream; after close the plan is owned by nobody
 * ---------------------------------------------------------------------------------------------------------------- */
size_t tpdm_stream_workspace_bytes(const tpdm_plan* plan, int capacity);
/* workspace: 1 KiB aligned, >= tpdm_stream_workspace_bytes; borrowed until tpdm_stream_close.  Encodes the TMA maps of the
 * stream's own context_embedder GEMM (2 * batch rows of staging). */
int tpdm_stream_open(tpdm_plan* plan, int capacity, float guidance_scale, void* workspace, size_t workspace_bytes, void* stream);
/* Admit n prompts into the free entries entry_ids[n] (host array, each in [0, capacity)): latents [n][C][h][w],
 * *_embeds [n][T][joint_attention_dim], *_pooled [n][pooled_projection_dim], device fp32, read by the enqueued work only.
 * Runs `batch` prompts per pass through the stream's own staging (text cast, context_embedder, pooled-text MLP), copies them
 * into their entries, publishes them, then lets idle slots claim: a prompt submitted to an idle stream runs in the next step.
 * Every prompt gets the stream's defaults: the guidance given to tpdm_stream_open, the plan's max_steps, predict = 1. */
int tpdm_stream_submit(tpdm_plan* plan, int n, const int* entry_ids, const float* latents, const float* neg_embeds,
                       const float* pos_embeds, const float* neg_pooled, const float* pos_pooled, void* stream);
/* Options of one request.  Invalid options (non-finite guidance, max_steps outside [1, plan max_steps], predict other than 0 / 1,
 * reserved != 0) make tpdm_stream_submit_options return TPDM_ERR_ARG before anything is enqueued. */
typedef struct tpdm_request_options {
  float guidance_scale;   /* finite */
  int32_t max_steps;      /* 1 .. plan max_steps */
  int32_t predict;        /* 1 = Beta mode, 0 = Beta draw from `seed` */
  int32_t reserved;       /* 0 */
  uint64_t seed;
} tpdm_request_options;   /* 24 bytes */
/* tpdm_stream_submit with options[n] (host array; NULL = the stream's defaults for every prompt) */
int tpdm_stream_submit_options(tpdm_plan* plan, int n, const int* entry_ids, const float* latents, const float* neg_embeds,
                               const float* pos_embeds, const float* neg_pooled, const float* pos_pooled,
                               const tpdm_request_options* options, void* stream);
/* device pointers: counters int[4] followed by `active` (slots holding a prompt) and the skip flag; done_log int[capacity]
 * (entry ids in completion order, entry k of the log at k % capacity); per entry: out_latents [capacity][C][h][w],
 * out_steps [capacity], out_sigmas [capacity][max_steps + 1].  A completion counted after a step is readable once that
 * step has completed. */
int tpdm_stream_status(tpdm_plan* plan, const int** counters, const int** done_log, const float** out_latents, const int** out_steps,
                       const float** out_sigmas);
/* device pointers [capacity][max_steps]: per-entry alpha, beta, raw log-prob of each executed step (step k of an entry's
 * request at [entry][k], k < its out_steps; later elements are not written).  Readable like the other outputs of an entry. */
int tpdm_stream_records(tpdm_plan* plan, const float** alphas, const float** betas, const float** logprobs);
/* Detach the stream (the caller synchronises first); the plan can then begin a queue or open a new stream. */
int tpdm_stream_close(tpdm_plan* plan);

/* ----------------------------------------------------------------------------------------------------------------
 * VAE decode of the final latent (SURVEY.md 8(f) rank 1).  Replaces, for the decode step only,
 *   latents = latents / vae.config.scaling_factor + vae.config.shift_factor
 *   image   = vae.decode(latents, return_dict=False)[0];  image_processor.postprocess(image, "pil")
 * (/root/reference/src/models/stable_diffusion_3/modeling_sd3_pnt.py:631, 653-655; AutoencoderKL is a diffusers class,
 * the decoder topology restated here is documented in DESIGN.md section 7).
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct tpdm_vae_config {
  int latent_channels;        /* 16 for SD3 (<= 64) */
  int out_channels;           /* 3 (<= 4) */
  int num_levels;             /* len(block_out_channels), <= 8 */
  int block_out_channels[8];  /* encoder order, e.g. 128, 256, 512, 512; each a multiple of 64 and of 4*norm_num_groups */
  int layers_per_block;       /* 2: every up block has layers_per_block + 1 resnets */
  int norm_num_groups;        /* 32 */
  float scaling_factor;       /* 1.5305 */
  float shift_factor;         /* 0.0609 */
} tpdm_vae_config;

/* 3x3 conv weights: bf16 [Cout][9][Cin] (tap = ky*3 + kx, then input channel); 1x1 / linear weights: bf16 [Cout][Cin];
 * biases and GroupNorm affine parameters fp32.  All pointers are device pointers borrowed for the lifetime of the ctx. */
typedef struct tpdm_vae_resnet {
  const float *norm1_w, *norm1_b;
  const void* conv1_w;
  const float* conv1_b;
  const float *norm2_w, *norm2_b;
  const void* conv2_w;
  const float* conv2_b;
  const void* short_w;        /* conv_shortcut (1x1), NULL when Cin == Cout */
  const float* short_b;
} tpdm_vae_resnet;

typedef struct tpdm_vae_weights {
  const void* conv_in_w;      /* bf16 [C0][9][64]: latent channels zero-padded to 64 */
  const float* conv_in_b;
  const tpdm_vae_resnet* resnets; /* mid_block.resnets.0, .1, then up_blocks.{i}.resnets.{j} in order */
  int n_resnets;              /* = tpdm_vae_num_resnets() */
  const float *attn_norm_w, *attn_norm_b; /* mid_block.attentions.0.group_norm */
  const void *attn_q_w, *attn_k_w, *attn_v_w, *attn_o_w;
  const float *attn_q_b, *attn_k_b, *attn_v_b, *attn_o_b;
  const void* const* up_conv_w; /* up_blocks.{i}.upsamplers.0.conv, i < num_levels - 1 */
  const float* const* up_conv_b;
  int n_upsamplers;
  const float *norm_out_w, *norm_out_b;   /* conv_norm_out */
  const void* conv_out_w;     /* bf16 [8][9][C_last]: rows >= out_channels are zero */
  const float* conv_out_b;    /* fp32 [8] */
} tpdm_vae_weights;

typedef struct tpdm_vae tpdm_vae;
int tpdm_vae_create(const tpdm_vae_config* cfg, tpdm_vae** out);
int tpdm_vae_destroy(tpdm_vae* vae);
int tpdm_vae_num_resnets(const tpdm_vae* vae);
int tpdm_vae_set_weights(tpdm_vae* vae, const tpdm_vae_weights* w);
/* bytes for one decode of a latent_h x latent_w latent (samples of a batch are decoded one after the other) */
size_t tpdm_vae_workspace_bytes(const tpdm_vae* vae, int latent_h, int latent_w);
/* latents fp32 NCHW [batch][latent_channels][h][w].  apply_scaling != 0: the input is the sampler's latent and
 * z = latents / scaling_factor + shift_factor is applied first (modeling_sd3_pnt.py:653); 0: the input is already z (what
 * AutoencoderKL.decode takes).  Outputs (either may be NULL, not both):
 * image fp32 NCHW [batch][out_channels][H][W] (what vae.decode returns), rgb uint8 [batch][H][W][out_channels] =
 * round(clamp(image / 2 + 0.5, 0, 1) * 255) (VaeImageProcessor.postprocess up to the PIL wrapper).  H = h * 2^(levels-1).
 * workspace: 1 KiB aligned, >= tpdm_vae_workspace_bytes().  Stream-ordered, no host synchronisation. */
int tpdm_vae_decode(tpdm_vae* vae, const float* latents, int apply_scaling, int batch, int latent_h, int latent_w,
                    void* workspace, size_t workspace_bytes, float* image, unsigned char* rgb, void* stream);

/* kernels launched by this library in this process since the last reset */
long long tpdm_launch_count(int reset);
/* bracket every GEMM (class 0) and attention (class 1) launch with CUDA events on the launching stream until stop;
 * stop returns, per class, the summed device time (ms), the algorithmic FLOPs and the number of launches */
int tpdm_profile_start(int max_records);
int tpdm_profile_stop(double* ms, double* flops, long long* count, int n_classes);
/* launches of the last tpdm_profile_stop that were left out because the device skipped them (a denoising step enqueued
 * speculatively after the trajectory had ended, see tpdm_sample_step): they did no work and are credited no FLOPs */
long long tpdm_profile_dropped(void);

/* ---- unit entry points used by tests/ (one kernel each) ---------------------------------------------------------- */
/* out = epilogue(A[batch][rows][K] (bf16) . W[N][K]^T (bf16)); epi: 0 bias->bf16, 1 bias->f32, 2 bias+gelu->bf16,
 * 3 out(f32) += gate[batch][N] * (acc + bias) */
int tpdm_gemm_bf16(const void* A, const void* W, const float* bias, const float* gate, void* out, int batch, int rows,
                   int N, int K, int epi, void* stream);
/* qkv bf16 [Bt][S][3*H*dp] -> out bf16 [Bt][S][H*dp] */
int tpdm_joint_attention(const void* qkv, void* out, int Bt, int S, int H, int dp, int head_dim, int q_rows, void* stream);
/* Diagnostic (synchronises the device): how many 128-row query tiles of the LAST attention launch were recomputed with the exact
 * softmax (scores more than ~2^64 above everything their row had seen before); -1 when the launch had no flag buffer (its
 * allocation failed).  0 on ordinary activations. */
int tpdm_attention_redo_count(void);
/* the same, summed over every attention launch since the library was loaded */
long long tpdm_attention_redo_total(void);
/* conv3x3 pad 1 over NHWC bf16 x [batch][g][g][C], w bf16 [N][9][C] -> out fp32 [batch][g*g][N] */
int tpdm_conv3x3_nhwc(const void* x, const void* w, const float* bias, float* out, int batch, int g, int C, int N,
                      void* stream);
/* conv3x3 (pad 1) weight gradient: dyt bf16 [samples][M][g*g], x bf16 three x-shifted NCHW copies [samples][3][C][g][g]
 * (copy k = X[..., x + k - 1], zero outside) -> dw fp32 [M][9][C] */
int tpdm_conv3x3_wgrad(const void* dyt, const void* x_shifted_nchw, float* dw, int samples, int g, int C, int M, void* stream);
/* LayerNorm(eps 1e-6, no affine) * (1 + scale[b]) + shift[b] : x fp32 [batch][rows][D] -> bf16 */
int tpdm_ln_modulate(const float* x, const float* shift, const float* scale, int mod_stride, void* out_bf16, int batch,
                     int rows, int D, void* stream);
/* tpdm_ln_modulate over two segments in ONE launch, the form every MMDiT block runs for its image and text rows: segment i
 * is x_i fp32 [batch][rows_i][D] -> out_i bf16, modulated by shift_i / scale_i (batch entry b at + b * mod_stride).  For tests of
 * that launch; the blocks reach the same launch internally. */
int tpdm_ln_modulate_pair(const float* x0, const float* shift0, const float* scale0, void* out0_bf16, int rows0, const float* x1,
                          const float* shift1, const float* scale1, void* out1_bf16, int rows1, int mod_stride, int batch, int D,
                          void* stream);
/* E4M3 row quantization, the rounding every FP8 operand of the library uses: per row, amax = max |x|, codes =
 * cvt.rn.satfinite.e4m3(x * (448 / amax)), scale = amax / 448 (IEEE fp32 divisions), so x ~= code * scale; a zero row gets
 * scale 1 and zero codes.  x fp32 [rows][K] (K % 4 == 0) -> codes E4M3 [rows][K], scales fp32 [rows]. */
int tpdm_quantize_fp8_rows(const float* x, int rows, int K, void* codes, float* scales, void* stream);
/* tpdm_ln_modulate with the result quantized per row as above: codes E4M3 [batch][rows][D], scales fp32 [batch][rows] */
int tpdm_ln_modulate_fp8(const float* x, const float* shift, const float* scale, int mod_stride, void* out_codes, float* out_scales,
                         int batch, int rows, int D, void* stream);
/* out = epilogue((A8[batch][rows][K] . W8[N][K]^T) * a_scale[batch][rows] * w_scale[N] + bias), E4M3 operands, fp32
 * accumulation; epi 0 -> bf16, 1 -> f32, 2 gelu -> bf16.  N > 128, K % 16 == 0. */
int tpdm_gemm_fp8(const void* A8, const float* a_scale, const void* W8, const float* w_scale, const float* bias, void* out, int batch,
                  int rows, int N, int K, int epi, void* stream);
/* Launch guards of the calling thread, the two the device-side prompt queue uses: when *skip_flag != 0 (device int) every
 * guarded launch returns at once; batch entry b of a launch is skipped when slot_active[b % slots] == 0 (device int[slots]).
 * They apply to every later launch of this library on the thread -- plan calls included -- until they are cleared with
 * (NULL, NULL, 1).  tpdm_queue_step clears both when it returns; tpdm_sample_step clears only the skip flag.  Guarded: the GEMMs
 * (both kernels, bf16 and E4M3), attention and ln_modulate (bf16 and E4M3).  slots < 1 is TPDM_ERR_ARG. */
int tpdm_set_launch_guards(const int* skip_flag, const int* slot_active, int slots);
/* One op of tpdm_gemm_ops: out = epilogue(A . W^T) as in tpdm_gemm_bf16, with free strides.  Element (b, r, k) of A is at
 * A + b * a_batch_stride + r * a_row_stride + k; output element (b, r, n) at out + b * out_batch_stride + r * ldo + n; the gate of
 * epi 3 at gate + b * gate_stride + n (strides in elements).  a_scale / w_scale both set: A and W are E4M3 codes with row
 * scales [batch][rows] and channel scales [N] (epi 0-2, N > 128; see tpdm_gemm_fp8); one of them alone is TPDM_ERR_ARG.
 * ksplit > 1: K is cut into ksplit ranges of ceil(nkb / ksplit) 64-wide k-blocks (nkb = ceil(K / 64)); range s writes its
 * partial product to out + (s * batch + b) * out_batch_stride (bias-free epi 1 with N <= 128 only). */
typedef struct tpdm_gemm_op_desc {
  const void* A;
  int64_t a_row_stride;
  int64_t a_batch_stride;
  const void* W;
  void* out;
  int64_t out_batch_stride;
  const float* bias;     /* [N] or NULL */
  const float* gate;     /* epi 3 only */
  const float* a_scale;  /* E4M3 operands only */
  const float* w_scale;
  int32_t rows;
  int32_t batch;
  int32_t K;
  int32_t N;
  int32_t epi;           /* 0 bias->bf16, 1 bias->f32, 2 bias+gelu->bf16, 3 out(f32) += gate * (acc + bias) */
  int32_t ldo;
  int32_t gate_stride;
  int32_t ksplit;        /* 1 = no split */
} tpdm_gemm_op_desc;
/* One persistent GEMM launch over n_ops (1 or 2) ops, the grouped form the MMDiT blocks use for the image and text streams. */
int tpdm_gemm_ops(const tpdm_gemm_op_desc* ops, int n_ops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TPDM_B200_H_ */
