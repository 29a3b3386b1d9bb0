// tpdm_b200 -- C ABI: context, plan (shape-bound workspace + prebuilt TMA descriptors) and the step orchestration.
// One tpdm_sample_step = MMDiT forward -> CFG -> TimePredictor -> schedule update -> Euler, enqueued on one stream with
// no host synchronisation (replaces the body of the loop at
// /root/reference/src/models/stable_diffusion_3/modeling_sd3_pnt.py:522-612).
#include <string.h>

#include <new>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "host.h"
#include "kernels.h"

using namespace tpdm;

struct tpdm_ctx {
  tpdm_config cfg;
  tpdm_weights w;
  std::vector<tpdm_block_weights> blocks;
  bool has_weights = false, has_mmdit = false, has_tpm = false;
  int D = 0, dp = 0, Dp = 0, R = 0, device = 0;
  std::vector<int> mod_off;  // first adaLN row of block i (norm1 rows, then norm1_context rows)
  bool any_dual = false;
  std::vector<tpdm_fp8_block_weights> fp8;  // tpdm_set_fp8_weights; empty = bf16 everywhere
  bool planned = false;                     // a plan was created: the GEMM operand types are fixed from then on
  bool dual(int i) const { return i < 64 && ((cfg.dual_attention_mask >> i) & 1ull) != 0; }
  int norm1_rows(int i) const { return (dual(i) ? 9 : 6) * D; }
};

namespace {

struct BlockOps {
  GemmOp qkv[2], out[2], ff1[2], ff2[2];
  AttnOp attn;
  int n_streams;  // 2, or 1 for the last (context_pre_only) block
  bool dual = false;  // SD3.5 dual-attention block: attn2 over the image tokens
  GemmOp qkv2, out2;
  AttnOp attn2;
};

struct Carver {
  uint8_t* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<uint8_t*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 1023) & ~size_t(1023);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

// which driver owns the plan's buffers: the lockstep sampler, the closed prompt queue or the open prompt stream
enum class Mode { kIdle, kSample, kQueue, kStream };

// one captured step and the launches it replays
struct StepGraph {
  cudaGraphExec_t exec = nullptr;
  long long launches = 0;
  StepGraph() = default;
  StepGraph(const StepGraph&) = delete;
  StepGraph& operator=(StepGraph&& o) noexcept {  // the moved-from graph destroys what this one held
    std::swap(exec, o.exec);
    std::swap(launches, o.launches);
    return *this;
  }
  void drop() {
    if (exec) cudaGraphExecDestroy(exec);
    exec = nullptr;
    launches = 0;
  }
  ~StepGraph() { drop(); }
};

}  // namespace

struct tpdm_plan {
  tpdm_ctx* ctx = nullptr;
  int B = 0, cfg_pairs = 0, Bt = 0, Hl = 0, Wl = 0, g = 0, N = 0, T = 0, S = 0, max_steps = 0;
  // MMDiT activations
  float *x_img, *x_ctx, *ctx0, *mod, *temb, *tproj, *thid, *text_part, *phid, *pout;
  bf16 *xn_img, *xn_ctx, *qkv, *attn_o, *ff_img, *ff_ctx, *enc_bf16;
  bf16 *xn2_img = nullptr, *qkv2 = nullptr, *attn_o2 = nullptr;  // dual-attention blocks only
  uint8_t *xn8_img = nullptr, *xn8_ctx = nullptr;  // FP8 mode: E4M3 QKV / FF1 inputs and their row scales
  float *xs_img = nullptr, *xs_ctx = nullptr;
  // TimePredictor
  bf16* tpm_x;
  float *y1, *y1p, *a2, *y2, *tpm_emb, *temb_cfg, *alpha_beta;
  int conv1_split = 1;  // split-K factor of TimePredictor.conv1 (few M tiles, K = 9 * 2D)
  double* gn_stats;
  // sampling state
  float *latents, *velocity, *sigma_hist, *alphas, *betas, *logprobs, *tembs, *history, *ratios;
  int *masks, *all_done;
  float* row_guidance;  // [B] guidance scale of each batch row, read by every CFG combine
  int predict = 1, have_ratios = 0;
  Mode mode = Mode::kIdle;
  unsigned long long seed = 0;
  std::vector<BlockOps> blk;
  GemmOp ctx_embed, proj_out, conv1;
  // device-side prompt queue (tpdm_queue_*): the plan's batch entries are in-flight slots
  struct Queue {
    int n_prompts = 0;
    const float* noise_all = nullptr;
    float *ctx0_all = nullptr, *text_all = nullptr, *sigma_cur = nullptr, *sigma_next = nullptr, *out_latents = nullptr, *out_sigmas = nullptr;
    int *slot_prompt = nullptr, *slot_step = nullptr, *slot_flush = nullptr, *slot_load = nullptr, *slot_active = nullptr, *ticket = nullptr,
        *out_steps = nullptr, *active = nullptr, *idle_flag = nullptr;
    const int* order = nullptr;
    const float* init_sigma = nullptr;
    int init_step = 0, n_queued = 0;
    // sampled rollouts (tpdm_queue_set_rollout); tpdm_queue_begin resets the queue to predict mode
    int predict = 1;
    unsigned long long seed = 0;
    const float* ratios_all = nullptr;
    float *rec_alphas = nullptr, *rec_betas = nullptr, *rec_logprobs = nullptr, *rec_tembs = nullptr;
    bf16* rec_tpm = nullptr;
    StepGraph graph;   // one captured queue step (every pointer of a queue step is fixed between steps)
  } q;
  // open prompt stream (tpdm_stream_*): the queue above runs over a ring of `capacity` entries, prompts are admitted between steps
  struct Stream {
    int capacity = 0;
    float guidance = 7.0f;   // the options of a request submitted without its own
    int *order = nullptr, *counters = nullptr, *done_log = nullptr;
    float* noise = nullptr;
    // request options [capacity] and per-step records [capacity][max_steps] of each entry
    float* guidance_all = nullptr;
    int *max_steps_all = nullptr, *predict_all = nullptr;
    unsigned long long* seed_all = nullptr;
    float *rec_alphas = nullptr, *rec_betas = nullptr, *rec_logprobs = nullptr;
    // admission staging, never read by a queue step: bf16 text [2*slots][T][J] (row 2k + half), its context_embedder output and
    // the pooled-text MLP of the same rows
    bf16* enc = nullptr;
    float *ctx0 = nullptr, *phid = nullptr, *text = nullptr;
    GemmOp ctx_embed;
  } st;
  // tpdm_sample_step_graph: one captured graph per step index (the step index only moves pointers inside the plan's own buffers),
  // valid for the predict / injected-ratio setting they were captured under (the guidance is read from row_guidance)
  std::vector<StepGraph> step_graph;
  int graph_predict = -1, graph_have_ratios = -1;
};

namespace {

constexpr unsigned in(Mode m) { return 1u << static_cast<int>(m); }

// TPDM_ERR_STATE unless the plan is in one of the `allowed` modes (a mask of in(Mode)); the message says what comes first
int check_mode(const tpdm_plan* p, unsigned allowed, const char* who) {
  if (allowed & in(p->mode)) return 0;
  const char* why = p->mode == Mode::kStream        ? "the plan has an open prompt stream (tpdm_stream_close first)"
                    : allowed == in(Mode::kSample)  ? "call tpdm_sample_begin first"
                    : allowed & in(Mode::kQueue)    ? "call tpdm_queue_begin first"
                    : allowed == in(Mode::kStream)  ? "the plan has no open stream"
                                                    : "a prompt queue runs on this plan";
  return fail(TPDM_ERR_STATE, "%s: %s", who, why);
}

// Replays g, capturing it from enqueue(stream) on first use.  The launch counters count a replay like the plain launches.
template <typename F>
int replay_or_capture(StepGraph& g, cudaStream_t s, const char* who, F enqueue) {
  if (g.exec == nullptr) {
    const long long before = launches_so_far();
    cudaGraph_t graph = nullptr;
    TPDM_CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const int st = enqueue(s);
    const cudaError_t e = cudaStreamEndCapture(s, &graph);
    if (st != 0) {
      if (graph) cudaGraphDestroy(graph);
      return st;
    }
    TPDM_CHECK(e == cudaSuccess && graph != nullptr, TPDM_ERR_CUDA, "%s: stream capture failed: %s", who, cudaGetErrorString(e));
    const cudaError_t ei = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    TPDM_CHECK(ei == cudaSuccess, TPDM_ERR_CUDA, "%s: cudaGraphInstantiate failed: %s", who, cudaGetErrorString(ei));
    g.launches = launches_so_far() - before;
    count_launches(-g.launches);  // the capture itself launched nothing
  }
  TPDM_CUDA_OK(cudaGraphLaunch(g.exec, s));
  count_launches(g.launches);
  return 0;
}

void set_shape(tpdm_plan* p, int batch, int cfg_pairs, int latent_h, int latent_w, int n_text, int max_steps) {
  p->B = batch;
  p->cfg_pairs = cfg_pairs ? 1 : 0;
  p->Bt = cfg_pairs ? 2 * batch : batch;
  p->Hl = latent_h;
  p->Wl = latent_w;
  p->g = latent_w / 2;
  p->N = p->g * p->g;
  p->T = n_text;
  p->S = p->N + p->T;
  p->max_steps = max_steps;
}

void carve(tpdm_plan* p, Carver& c) {
  const tpdm_ctx* ctx = p->ctx;
  const size_t Bt = p->Bt, B = p->B, N = p->N, T = p->T, S = p->S, D = ctx->D, Dp = ctx->Dp, R = ctx->R;
  const size_t C1 = ctx->cfg.tpm_channels, g = p->g, steps = p->max_steps;
  const size_t lat = static_cast<size_t>(ctx->cfg.in_channels) * p->Hl * p->Wl;
  p->x_img = c.take<float>(Bt * N * D);
  p->x_ctx = c.take<float>(Bt * T * D);
  p->ctx0 = c.take<float>(Bt * T * D);
  p->mod = c.take<float>(Bt * R);
  p->temb = c.take<float>(Bt * D);
  p->tproj = c.take<float>(Bt * 256);
  p->thid = c.take<float>(Bt * D);
  p->text_part = c.take<float>(Bt * D);
  p->phid = c.take<float>(Bt * D);
  p->pout = c.take<float>(Bt * N * 4 * ctx->cfg.out_channels);
  p->xn_img = c.take<bf16>(Bt * N * D);
  p->xn_ctx = c.take<bf16>(Bt * T * D);
  p->qkv = c.take<bf16>(Bt * S * 3 * Dp);
  p->attn_o = c.take<bf16>(Bt * S * Dp);
  if (ctx->any_dual) {
    p->xn2_img = c.take<bf16>(Bt * N * D);
    p->qkv2 = c.take<bf16>(Bt * N * 3 * Dp);
    p->attn_o2 = c.take<bf16>(Bt * N * Dp);
  }
  if (!ctx->fp8.empty()) {
    p->xn8_img = c.take<uint8_t>(Bt * N * D);
    p->xn8_ctx = c.take<uint8_t>(Bt * T * D);
    p->xs_img = c.take<float>(Bt * N);
    p->xs_ctx = c.take<float>(Bt * T);
  }
  p->ff_img = c.take<bf16>(Bt * N * 4 * D);
  p->ff_ctx = c.take<bf16>(Bt * T * 4 * D);
  p->enc_bf16 = c.take<bf16>(Bt * T * ctx->cfg.joint_attention_dim);
  p->tpm_x = c.take<bf16>(Bt * g * g * 2 * D);  // Bt (not B) rows so the stand-alone TPM entry point can take Bt samples
  p->y1 = c.take<float>(Bt * g * g * C1);
  p->y1p = c.take<float>(4 * Bt * g * g * C1);  // partial products of the split-K conv1
  p->a2 = c.take<float>(Bt * g * g * C1);
  p->y2 = c.take<float>(Bt * (g / 2) * (g / 2) * C1);
  p->tpm_emb = c.take<float>(Bt * 2 * C1);
  p->temb_cfg = c.take<float>(Bt * D);
  p->alpha_beta = c.take<float>(Bt * 2);
  p->gn_stats = c.take<double>(Bt * 2);
  p->latents = c.take<float>(B * lat);
  p->velocity = c.take<float>(B * lat);
  p->sigma_hist = c.take<float>(B * (steps + 1));
  p->alphas = c.take<float>(B * steps);
  p->betas = c.take<float>(B * steps);
  p->logprobs = c.take<float>(B * steps);
  p->ratios = c.take<float>(B * steps);
  p->masks = c.take<int>(B * steps);
  p->all_done = c.take<int>(steps);
  p->tembs = c.take<float>(steps * B * D);
  p->history = c.take<float>(steps * B * lat);
  p->row_guidance = c.take<float>(B);
}

int check_shapes(const tpdm_ctx* ctx, int batch, int latent_h, int latent_w, int n_text, int max_steps) {
  TPDM_CHECK(ctx != nullptr, TPDM_ERR_ARG, "null ctx");
  TPDM_CHECK(batch > 0 && n_text > 0 && max_steps > 0, TPDM_ERR_SHAPE, "batch, n_text and max_steps must be positive");
  TPDM_CHECK(latent_h == latent_w, TPDM_ERR_SHAPE, "only square latents are supported (got %dx%d)", latent_h, latent_w);
  const int g = latent_w / 2;
  TPDM_CHECK(latent_w % 2 == 0 && g >= 8 && g <= 128 && (g & (g - 1)) == 0, TPDM_ERR_SHAPE,
             "latent side %d: token grid side must be a power of two in [8,128]", latent_w);
  TPDM_CHECK(g <= ctx->cfg.pos_embed_max_size, TPDM_ERR_SHAPE, "token grid %d exceeds pos_embed_max_size %d", g,
             ctx->cfg.pos_embed_max_size);
  return 0;
}

int build_ops(tpdm_plan* p) {
  tpdm_ctx* ctx = p->ctx;
  const int D = ctx->D, Dp = ctx->Dp, R = ctx->R, L = ctx->cfg.num_layers;
  const int Bt = p->Bt, N = p->N, T = p->T, S = p->S;
  const tpdm_weights& w = ctx->w;
  if (ctx->has_tpm)
    {
      // conv1 has g*g/128 M tiles per sample and K = 9 * 2D: with one prompt in flight that is 32 CTAs walking 432 k-blocks each.
      // K is cut in 4 (deterministic partial products, summed with the bias by k_sum_partials) when it divides evenly.
      const int nkb = 9 * 2 * D / 64;
      p->conv1_split = nkb % 4 == 0 ? 4 : 1;
      if (p->conv1_split > 1) {
        TPDM_TRY(gemm_op_init_conv3x3(&p->conv1, p->tpm_x, Bt, p->g, 2 * D, w.tpm_conv1_w, ctx->cfg.tpm_channels, EPI_BIAS_F32, p->y1p,
                                      ctx->cfg.tpm_channels, nullptr));
        TPDM_TRY(gemm_op_set_ksplit(&p->conv1, p->conv1_split));
      } else {
        TPDM_TRY(gemm_op_init_conv3x3(&p->conv1, p->tpm_x, Bt, p->g, 2 * D, w.tpm_conv1_w, ctx->cfg.tpm_channels, EPI_BIAS_F32, p->y1,
                                      ctx->cfg.tpm_channels, w.tpm_conv1_b));
      }
    }
  if (!ctx->has_mmdit) return 0;
  p->blk.resize(L);
  for (int i = 0; i < L; ++i) {
    const tpdm_block_weights& bw = ctx->blocks[i];
    BlockOps& o = p->blk[i];
    const bool last = i == L - 1;
    o.n_streams = last ? 1 : 2;
    float* mod_img = p->mod + ctx->mod_off[i];
    float* mod_ctx = mod_img + ctx->norm1_rows(i);
    o.dual = ctx->dual(i);
    const bool fp8 = !ctx->fp8.empty();
    // fused QKV: image rows land at tokens [0,N), text rows at [N,S) of the joint qkv buffer
    if (fp8) {
      const tpdm_fp8_block_weights& fw = ctx->fp8[i];
      TPDM_TRY(gemm_op_init_fp8(&o.qkv[0], p->xn8_img, D, static_cast<long long>(N) * D, p->xs_img, N, Bt, D, fw.qkv_w, fw.qkv_s, 3 * Dp,
                                EPI_BIAS_BF16, p->qkv, static_cast<long long>(S) * 3 * Dp, 3 * Dp, bw.qkv_b));
      TPDM_TRY(gemm_op_init_fp8(&o.qkv[1], p->xn8_ctx, D, static_cast<long long>(T) * D, p->xs_ctx, T, Bt, D, fw.cqkv_w, fw.cqkv_s, 3 * Dp,
                                EPI_BIAS_BF16, p->qkv + static_cast<size_t>(N) * 3 * Dp, static_cast<long long>(S) * 3 * Dp, 3 * Dp, bw.cqkv_b));
    } else {
      TPDM_TRY(gemm_op_init(&o.qkv[0], p->xn_img, D, static_cast<long long>(N) * D, N, Bt, D, bw.qkv_w, 3 * Dp, EPI_BIAS_BF16, p->qkv,
                            static_cast<long long>(S) * 3 * Dp, 3 * Dp, bw.qkv_b, nullptr, 0));
      TPDM_TRY(gemm_op_init(&o.qkv[1], p->xn_ctx, D, static_cast<long long>(T) * D, T, Bt, D, bw.cqkv_w, 3 * Dp, EPI_BIAS_BF16,
                            p->qkv + static_cast<size_t>(N) * 3 * Dp, static_cast<long long>(S) * 3 * Dp, 3 * Dp, bw.cqkv_b, nullptr, 0));
    }
    TPDM_TRY(attn_op_init(&o.attn, p->qkv, Bt, S, ctx->cfg.num_heads, ctx->dp, ctx->cfg.head_dim, p->attn_o));
    if (last) o.attn.q_tiles = (N + 127) / 128;  // context_pre_only: text-query rows are never used
    // output projections: x += gate_msa * (o W^T + b)
    TPDM_TRY(gemm_op_init(&o.out[0], p->attn_o, Dp, static_cast<long long>(S) * Dp, N, Bt, Dp, bw.out_w, D, EPI_GATE_RESIDUAL, p->x_img,
                          static_cast<long long>(N) * D, D, bw.out_b, mod_img + 2 * D, R));
    if (fp8)
      TPDM_TRY(gemm_op_init_fp8(&o.ff1[0], p->xn8_img, D, static_cast<long long>(N) * D, p->xs_img, N, Bt, D, ctx->fp8[i].ff1_w, ctx->fp8[i].ff1_s,
                                4 * D, EPI_BIAS_GELU_BF16, p->ff_img, static_cast<long long>(N) * 4 * D, 4 * D, bw.ff1_b));
    else
      TPDM_TRY(gemm_op_init(&o.ff1[0], p->xn_img, D, static_cast<long long>(N) * D, N, Bt, D, bw.ff1_w, 4 * D, EPI_BIAS_GELU_BF16,
                            p->ff_img, static_cast<long long>(N) * 4 * D, 4 * D, bw.ff1_b, nullptr, 0));
    TPDM_TRY(gemm_op_init(&o.ff2[0], p->ff_img, 4 * D, static_cast<long long>(N) * 4 * D, N, Bt, 4 * D, bw.ff2_w, D, EPI_GATE_RESIDUAL,
                          p->x_img, static_cast<long long>(N) * D, D, bw.ff2_b, mod_img + 5 * D, R));
    if (o.dual) {
      // SD3.5 attn2: self-attention over the image tokens from the second modulated copy of LN(x); x += gate_msa2 * (...)
      TPDM_CHECK(bw.qkv2_w && bw.qkv2_b && bw.out2_w && bw.out2_b, TPDM_ERR_ARG, "block %d: dual-attention block without attn2 weights", i);
      TPDM_TRY(gemm_op_init(&o.qkv2, p->xn2_img, D, static_cast<long long>(N) * D, N, Bt, D, bw.qkv2_w, 3 * Dp, EPI_BIAS_BF16, p->qkv2,
                            static_cast<long long>(N) * 3 * Dp, 3 * Dp, bw.qkv2_b, nullptr, 0));
      TPDM_TRY(attn_op_init(&o.attn2, p->qkv2, Bt, N, ctx->cfg.num_heads, ctx->dp, ctx->cfg.head_dim, p->attn_o2));
      TPDM_TRY(gemm_op_init(&o.out2, p->attn_o2, Dp, static_cast<long long>(N) * Dp, N, Bt, Dp, bw.out2_w, D, EPI_GATE_RESIDUAL, p->x_img,
                            static_cast<long long>(N) * D, D, bw.out2_b, mod_img + 8 * D, R));
    }
    if (!last) {
      TPDM_CHECK(bw.cout_w && bw.cff1_w && bw.cff2_w, TPDM_ERR_ARG, "block %d: missing context-stream weights", i);
      TPDM_TRY(gemm_op_init(&o.out[1], p->attn_o + static_cast<size_t>(N) * Dp, Dp, static_cast<long long>(S) * Dp, T, Bt, Dp, bw.cout_w,
                            D, EPI_GATE_RESIDUAL, p->x_ctx, static_cast<long long>(T) * D, D, bw.cout_b, mod_ctx + 2 * D, R));
      if (fp8)
        TPDM_TRY(gemm_op_init_fp8(&o.ff1[1], p->xn8_ctx, D, static_cast<long long>(T) * D, p->xs_ctx, T, Bt, D, ctx->fp8[i].cff1_w,
                                  ctx->fp8[i].cff1_s, 4 * D, EPI_BIAS_GELU_BF16, p->ff_ctx, static_cast<long long>(T) * 4 * D, 4 * D, bw.cff1_b));
      else
        TPDM_TRY(gemm_op_init(&o.ff1[1], p->xn_ctx, D, static_cast<long long>(T) * D, T, Bt, D, bw.cff1_w, 4 * D, EPI_BIAS_GELU_BF16,
                              p->ff_ctx, static_cast<long long>(T) * 4 * D, 4 * D, bw.cff1_b, nullptr, 0));
      TPDM_TRY(gemm_op_init(&o.ff2[1], p->ff_ctx, 4 * D, static_cast<long long>(T) * 4 * D, T, Bt, 4 * D, bw.cff2_w, D,
                            EPI_GATE_RESIDUAL, p->x_ctx, static_cast<long long>(T) * D, D, bw.cff2_b, mod_ctx + 5 * D, R));
    }
  }
  const int J = ctx->cfg.joint_attention_dim;
  TPDM_TRY(gemm_op_init(&p->ctx_embed, p->enc_bf16, J, static_cast<long long>(T) * J, T, Bt, J, w.ctx_w, D, EPI_BIAS_F32, p->ctx0,
                        static_cast<long long>(T) * D, D, w.ctx_b, nullptr, 0));
  const int PO = 4 * ctx->cfg.out_channels;
  TPDM_TRY(gemm_op_init(&p->proj_out, p->xn_img, D, static_cast<long long>(N) * D, N, Bt, D, w.proj_w, PO, EPI_BIAS_F32, p->pout,
                        static_cast<long long>(N) * PO, PO, w.proj_b, nullptr, 0));
  return 0;
}

// sigma-independent part: bf16 cast of the text embeddings, context_embedder GEMM, pooled-text MLP
// (transformer_sd3.py:337 and the text_embedder half of :336 -- hoisted out of the step loop).
int set_prompts(tpdm_plan* p, const float* enc_a, const float* enc_b, const float* pooled_a, const float* pooled_b, cudaStream_t s) {
  const tpdm_ctx* ctx = p->ctx;
  const tpdm_weights& w = ctx->w;
  const int D = ctx->D, J = ctx->cfg.joint_attention_dim, PD = ctx->cfg.pooled_projection_dim;
  const int half = enc_b ? p->B : p->Bt;
  const long long ne = static_cast<long long>(half) * p->T * J;
  TPDM_TRY(k_cast_bf16(enc_a, p->enc_bf16, ne, s));
  if (enc_b) TPDM_TRY(k_cast_bf16(enc_b, p->enc_bf16 + ne, ne, s));
  TPDM_TRY(gemm_launch(&p->ctx_embed, 1, s));
  TPDM_TRY(k_gemv_f32(w.p_w1, w.p_b1, pooled_a, PD, nullptr, p->phid, D, half, D, PD, 0, s));
  if (pooled_b) TPDM_TRY(k_gemv_f32(w.p_w1, w.p_b1, pooled_b, PD, nullptr, p->phid + static_cast<size_t>(half) * D, D, half, D, PD, 0, s));
  TPDM_TRY(k_gemv_f32(w.p_w2, w.p_b2, p->phid, D, nullptr, p->text_part, D, p->Bt, D, D, 1, s));
  return 0;
}

// FP8 mode: the LN-modulate feeding QKV / FF1 writes E4M3 rows + row scales (image stream seg[0], text stream seg[1])
void set_fp8_out(const tpdm_plan* p, LnSeg (&seg)[2]) {
  if (p->xn8_img == nullptr) return;
  seg[0].out8 = p->xn8_img;
  seg[0].out_scale = p->xs_img;
  seg[1].out8 = p->xn8_ctx;
  seg[1].out_scale = p->xs_ctx;
}

// CustomSD3Transformer2DModel.forward minus the sigma-independent part
int run_mmdit(tpdm_plan* p, const float* latents, int Bl, int dup, const float* timestep, int t_stride, float t_scale, int t_rep,
              float* h1_out, float* h2_out, bool tpm_taps, cudaStream_t s) {
  const tpdm_ctx* ctx = p->ctx;
  const tpdm_weights& w = ctx->w;
  const int D = ctx->D, R = ctx->R, L = ctx->cfg.num_layers, Bt = p->Bt, N = p->N, T = p->T;
  // temb = timestep MLP + hoisted pooled-text MLP, then every adaLN modulation vector of the step in one GEMV
  TPDM_TRY(k_timestep_embedding(timestep, t_stride, t_scale, p->tproj, Bt, t_rep, s));
  TPDM_TRY(k_gemv_f32(w.t_w1, w.t_b1, p->tproj, 256, nullptr, p->thid, D, Bt, D, 256, 0, s));
  TPDM_TRY(k_gemv_f32(w.t_w2, w.t_b2, p->thid, D, p->text_part, p->temb, D, Bt, D, D, 1, s));
  // (Measured and rejected: running the rows of blocks 1..L-1 on a side stream underneath block 0.  With 8-warp blocks the
  // GEMV cannot co-reside with a GEMM / attention CTA and nothing overlaps; with 4-warp blocks it does co-reside and the
  // step got 5-8 % SLOWER -- the resident GEMV blocks delay the CTAs of the tensor-core kernels.)
  TPDM_TRY(k_gemv_bf16(reinterpret_cast<const bf16*>(w.adaln_w), w.adaln_b, p->temb, D, nullptr, p->mod, R, Bt, R, D, 1, s));
  TPDM_TRY(k_patchify(latents, w.patch_w, w.patch_b, w.pos_table, ctx->cfg.pos_embed_max_size, p->x_img, Bl, dup, ctx->cfg.in_channels,
                      p->Hl, p->Wl, D, h1_out, tpm_taps ? p->tpm_x : nullptr, s));
  TPDM_CUDA_OK(cudaMemcpyAsync(p->x_ctx, p->ctx0, static_cast<size_t>(Bt) * T * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  for (int i = 0; i < L; ++i) {
    BlockOps& o = p->blk[i];
    const tpdm_block_weights& bw = ctx->blocks[i];
    const bool last = i == L - 1;
    const float* mi = p->mod + ctx->mod_off[i];
    const float* mc = mi + ctx->norm1_rows(i);
    LnSeg seg[2];
    seg[0] = LnSeg{p->x_img, p->xn_img, mi, mi + D, N, Bt, R};
    // last block: AdaLayerNormContinuous chunk order is (scale, shift)
    seg[1] = last ? LnSeg{p->x_ctx, p->xn_ctx, mc + D, mc, T, Bt, R} : LnSeg{p->x_ctx, p->xn_ctx, mc, mc + D, T, Bt, R};
    set_fp8_out(p, seg);
    TPDM_TRY(k_ln_modulate(seg, 2, D, s));
    if (o.dual) {  // norm_hidden_states2 = LN(x) * (1 + scale_msa2) + shift_msa2, from x BEFORE the first attention is added
      LnSeg seg2{p->x_img, p->xn2_img, mi + 6 * D, mi + 7 * D, N, Bt, R};
      TPDM_TRY(k_ln_modulate(&seg2, 1, D, s));
    }
    TPDM_TRY(gemm_launch(o.qkv, 2, s));
    if (ctx->cfg.qk_norm) {
      TPDM_TRY(k_qk_rmsnorm(p->qkv, Bt, p->S, 0, N, ctx->cfg.num_heads, ctx->dp, ctx->cfg.head_dim, bw.norm_q, bw.norm_k, s));
      TPDM_TRY(k_qk_rmsnorm(p->qkv, Bt, p->S, N, T, ctx->cfg.num_heads, ctx->dp, ctx->cfg.head_dim, bw.norm_added_q, bw.norm_added_k, s));
    }
    TPDM_TRY(attn_launch(&o.attn, s));
    TPDM_TRY(gemm_launch(o.out, o.n_streams, s));
    if (o.dual) {
      TPDM_TRY(gemm_launch(&o.qkv2, 1, s));
      if (ctx->cfg.qk_norm)
        TPDM_TRY(k_qk_rmsnorm(p->qkv2, Bt, N, 0, N, ctx->cfg.num_heads, ctx->dp, ctx->cfg.head_dim, bw.norm_q2, bw.norm_k2, s));
      TPDM_TRY(attn_launch(&o.attn2, s));
      TPDM_TRY(gemm_launch(&o.out2, 1, s));
    }
    seg[0] = LnSeg{p->x_img, p->xn_img, mi + 3 * D, mi + 4 * D, N, Bt, R};
    seg[1] = LnSeg{p->x_ctx, p->xn_ctx, mc + 3 * D, mc + 4 * D, T, Bt, R};
    set_fp8_out(p, seg);
    TPDM_TRY(k_ln_modulate(seg, o.n_streams, D, s));
    TPDM_TRY(gemm_launch(o.ff1, o.n_streams, s));
    TPDM_TRY(gemm_launch(o.ff2, o.n_streams, s));
  }
  const float* mno = p->mod + (R - 2 * D);  // norm_out rows: (scale, shift)
  const int pairs = tpm_taps ? p->cfg_pairs : 0;
  TPDM_TRY(k_norm_out(p->x_img, p->xn_img, mno + D, mno, R, pairs ? p->B : Bt, pairs, N, D, p->g, p->row_guidance,
                      tpm_taps ? p->tpm_x : nullptr, h2_out, s));
  TPDM_TRY(gemm_launch(&p->proj_out, 1, s));
  return 0;
}

// TimePredictor.forward on the NHWC bf16 tap buffer already in p->tpm_x
int run_tpm(tpdm_plan* p, int nb, const float* temb, float* alpha_beta, cudaStream_t s) {
  const tpdm_ctx* ctx = p->ctx;
  const tpdm_weights& w = ctx->w;
  const int C1 = ctx->cfg.tpm_channels, g = p->g, D = ctx->D;
  GemmOp conv = p->conv1;
  conv.batch = nb;
  conv.num_tiles = nb * conv.tiles_m_per_batch * conv.tiles_n * conv.ksplit;
  TPDM_TRY(gemm_launch(&conv, 1, s));
  if (conv.ksplit > 1)
    TPDM_TRY(k_sum_partials(p->y1p, conv.ksplit, static_cast<long long>(nb) * g * g * C1, w.tpm_conv1_b, C1, p->y1, s));
  TPDM_CUDA_OK(cudaMemsetAsync(p->gn_stats, 0, sizeof(double) * 2 * nb, s));
  TPDM_TRY(k_gn_stats(p->y1, p->gn_stats, nb, static_cast<long long>(g) * g * C1, s));
  TPDM_TRY(k_gemv_f32(w.tpm_lin_w, w.tpm_lin_b, temb, D, nullptr, p->tpm_emb, 2 * C1, nb, 2 * C1, D, 1, s));
  TPDM_TRY(k_gn_mod_silu(p->y1, p->gn_stats, w.tpm_gn_w, w.tpm_gn_b, p->tpm_emb, p->a2, nb, g * g, C1, s));
  TPDM_TRY(k_conv3x3_s2(p->a2, w.tpm_conv2_w, w.tpm_conv2_b, p->y2, nb, g, C1, s));
  TPDM_TRY(k_tpm_tail(p->y2, nb, g / 2, C1, w.tpm_fc1_w, w.tpm_fc1_b, w.tpm_fc2_w, w.tpm_fc2_b, ctx->cfg.tpm_epsilon, alpha_beta, s));
  return 0;
}

}  // namespace

// ==============================================================================================================
extern "C" {

int tpdm_create(const tpdm_config* cfg, tpdm_ctx** out) {
  TPDM_CHECK(cfg && out, TPDM_ERR_ARG, "tpdm_create: null argument");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  TPDM_CHECK(e == cudaSuccess && ndev > 0, TPDM_ERR_CUDA, "tpdm_create: no CUDA device (%s); this library has no CPU fallback",
             e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  int dev = 0;
  TPDM_CUDA_OK(cudaGetDevice(&dev));
  int major = 0;
  TPDM_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  TPDM_CHECK(major == 10, TPDM_ERR_CUDA, "tpdm_create: device compute capability %d.x; this library targets sm_100a only", major);
  TPDM_CHECK(cfg->patch_size == 2, TPDM_ERR_SHAPE, "patch_size %d unsupported (only 2)", cfg->patch_size);
  TPDM_CHECK(cfg->in_channels * 4 == 64 && cfg->out_channels * 4 == 64, TPDM_ERR_SHAPE, "in/out channels must be 16");
  TPDM_CHECK(cfg->head_dim > 0 && cfg->head_dim <= 128 && cfg->head_dim % 8 == 0, TPDM_ERR_SHAPE, "head_dim %d unsupported", cfg->head_dim);
  TPDM_CHECK(cfg->num_layers > 0 && cfg->num_heads > 0, TPDM_ERR_SHAPE, "empty model");
  TPDM_CHECK(cfg->tpm_channels > 0 && cfg->tpm_channels <= 128 && cfg->tpm_channels % 32 == 0, TPDM_ERR_SHAPE, "tpm_channels %d unsupported",
             cfg->tpm_channels);
  tpdm_ctx* c = new (std::nothrow) tpdm_ctx();
  TPDM_CHECK(c, TPDM_ERR_NOMEM, "out of host memory");
  c->cfg = *cfg;
  c->D = cfg->num_heads * cfg->head_dim;
  c->dp = cfg->head_dim <= 64 ? 64 : 128;
  c->Dp = cfg->num_heads * c->dp;
  TPDM_CHECK(cfg->num_layers <= 64 || cfg->dual_attention_mask == 0, TPDM_ERR_SHAPE, "dual_attention_mask covers 64 layers at most");
  TPDM_CHECK(cfg->num_layers >= 64 || (cfg->dual_attention_mask >> cfg->num_layers) == 0, TPDM_ERR_ARG,
             "dual_attention_mask names a layer >= num_layers");
  c->mod_off.resize(cfg->num_layers);
  int rows = 0;
  for (int i = 0; i < cfg->num_layers; ++i) {
    c->mod_off[i] = rows;
    rows += c->norm1_rows(i) + (i == cfg->num_layers - 1 ? 2 : 6) * c->D;
    c->any_dual = c->any_dual || c->dual(i);
  }
  c->R = rows + 2 * c->D;  // + norm_out
  c->device = dev;
  TPDM_CHECK(c->D % 64 == 0 && cfg->joint_attention_dim % 64 == 0, TPDM_ERR_SHAPE, "hidden sizes must be multiples of 64");
  *out = c;
  return 0;
}

int tpdm_destroy(tpdm_ctx* ctx) {
  delete ctx;
  return 0;
}

int tpdm_set_weights(tpdm_ctx* ctx, const tpdm_weights* w) {
  TPDM_CHECK(ctx && w, TPDM_ERR_ARG, "tpdm_set_weights: null argument");
  ctx->w = *w;
  ctx->has_mmdit = w->blocks != nullptr;
  ctx->has_tpm = w->tpm_conv1_w != nullptr;
  TPDM_CHECK(ctx->has_mmdit || ctx->has_tpm, TPDM_ERR_ARG, "tpdm_set_weights: neither MMDiT nor TimePredictor weights given");
  if (ctx->has_mmdit) {
    ctx->blocks.assign(w->blocks, w->blocks + ctx->cfg.num_layers);
    ctx->w.blocks = ctx->blocks.data();
    const void* req[] = {w->patch_w, w->patch_b, w->pos_table, w->t_w1, w->t_b1, w->t_w2, w->t_b2, w->p_w1, w->p_b1, w->p_w2, w->p_b2,
                         w->ctx_w, w->ctx_b, w->adaln_w, w->adaln_b, w->proj_w, w->proj_b};
    for (const void* p : req) TPDM_CHECK(p != nullptr, TPDM_ERR_ARG, "tpdm_set_weights: a required MMDiT weight pointer is null");
    for (int i = 0; i < ctx->cfg.num_layers; ++i) {
      const tpdm_block_weights& b = ctx->blocks[i];
      TPDM_CHECK(b.qkv_w && b.qkv_b && b.cqkv_w && b.cqkv_b && b.out_w && b.out_b && b.ff1_w && b.ff1_b && b.ff2_w && b.ff2_b, TPDM_ERR_ARG,
                 "tpdm_set_weights: block %d is missing weights", i);
      if (ctx->cfg.qk_norm)
        TPDM_CHECK(b.norm_q && b.norm_k && b.norm_added_q && b.norm_added_k, TPDM_ERR_ARG, "block %d: qk_norm weights missing", i);
      if (ctx->dual(i))
        TPDM_CHECK(b.qkv2_w && b.qkv2_b && b.out2_w && b.out2_b && (!ctx->cfg.qk_norm || (b.norm_q2 && b.norm_k2)), TPDM_ERR_ARG,
                   "block %d: dual-attention block is missing attn2 weights", i);
    }
  }
  if (ctx->has_tpm) {
    const void* req[] = {w->tpm_conv1_b, w->tpm_lin_w, w->tpm_lin_b, w->tpm_gn_w, w->tpm_gn_b, w->tpm_conv2_w, w->tpm_conv2_b,
                         w->tpm_fc1_w, w->tpm_fc1_b, w->tpm_fc2_w, w->tpm_fc2_b};
    for (const void* p : req) TPDM_CHECK(p != nullptr, TPDM_ERR_ARG, "tpdm_set_weights: a required TimePredictor weight pointer is null");
  }
  ctx->has_weights = true;
  return 0;
}

int tpdm_set_fp8_weights(tpdm_ctx* ctx, const tpdm_fp8_block_weights* blocks) {
  TPDM_CHECK(ctx && blocks, TPDM_ERR_ARG, "tpdm_set_fp8_weights: null argument");
  TPDM_CHECK(ctx->has_mmdit, TPDM_ERR_STATE, "tpdm_set_fp8_weights: call tpdm_set_weights with MMDiT weights first");
  TPDM_CHECK(!ctx->planned, TPDM_ERR_STATE, "tpdm_set_fp8_weights: a plan of this ctx already exists (set FP8 weights before the first plan)");
  const int L = ctx->cfg.num_layers;
  for (int i = 0; i < L; ++i) {
    const tpdm_fp8_block_weights& b = blocks[i];
    TPDM_CHECK(b.qkv_w && b.qkv_s && b.cqkv_w && b.cqkv_s && b.ff1_w && b.ff1_s && (i == L - 1 || (b.cff1_w && b.cff1_s)), TPDM_ERR_ARG,
               "tpdm_set_fp8_weights: block %d is missing FP8 weights or scales", i);
  }
  ctx->fp8.assign(blocks, blocks + L);
  return 0;
}

size_t tpdm_plan_workspace_bytes(const tpdm_ctx* ctx, int batch, int cfg_pairs, int latent_h, int latent_w, int n_text, int max_steps) {
  if (check_shapes(ctx, batch, latent_h, latent_w, n_text, max_steps) != 0) return 0;
  tpdm_plan p;
  p.ctx = const_cast<tpdm_ctx*>(ctx);
  set_shape(&p, batch, cfg_pairs, latent_h, latent_w, n_text, max_steps);
  Carver c(nullptr);
  carve(&p, c);
  return c.off + 1024;
}

int tpdm_plan_create(tpdm_ctx* ctx, int batch, int cfg_pairs, int latent_h, int latent_w, int n_text, int max_steps, void* workspace,
                     size_t workspace_bytes, tpdm_plan** out) {
  TPDM_CHECK(out && workspace, TPDM_ERR_ARG, "tpdm_plan_create: null argument");
  TPDM_TRY(check_shapes(ctx, batch, latent_h, latent_w, n_text, max_steps));
  TPDM_CHECK(ctx->has_weights, TPDM_ERR_STATE, "tpdm_plan_create: call tpdm_set_weights first");
  TPDM_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, TPDM_ERR_ARG, "workspace must be 1024-byte aligned");
  const size_t need = tpdm_plan_workspace_bytes(ctx, batch, cfg_pairs, latent_h, latent_w, n_text, max_steps);
  TPDM_CHECK(workspace_bytes >= need, TPDM_ERR_NOMEM, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  tpdm_plan* p = new (std::nothrow) tpdm_plan();
  TPDM_CHECK(p, TPDM_ERR_NOMEM, "out of host memory");
  p->ctx = ctx;
  set_shape(p, batch, cfg_pairs, latent_h, latent_w, n_text, max_steps);
  Carver c(workspace);
  carve(p, c);
  int st = build_ops(p);
  if (st != 0) {
    delete p;
    return st;
  }
  ctx->planned = true;
  *out = p;
  return 0;
}

int tpdm_plan_destroy(tpdm_plan* plan) {
  delete plan;
  return 0;
}

int tpdm_mmdit_forward(tpdm_plan* p, const float* latents, const float* timestep, const float* enc, const float* pooled, float* out_sample,
                       float* out_temb, float* out_h1, float* out_h2, void* stream) {
  TPDM_CHECK(p && latents && timestep && enc && pooled, TPDM_ERR_ARG, "tpdm_mmdit_forward: null argument");
  TPDM_CHECK(p->ctx->has_mmdit, TPDM_ERR_STATE, "tpdm_mmdit_forward: MMDiT weights were not set");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  TPDM_TRY(set_prompts(p, enc, nullptr, pooled, nullptr, s));
  TPDM_TRY(run_mmdit(p, latents, p->Bt, 1, timestep, 1, 1.0f, 1, out_h1, out_h2, false, s));
  if (out_sample)
    TPDM_TRY(k_unpatchify(p->pout, p->Bt, 0, p->row_guidance, ctx->cfg.out_channels, p->Hl, p->Wl, out_sample, nullptr, nullptr, nullptr, 0, nullptr, s));
  if (out_temb)
    TPDM_CUDA_OK(cudaMemcpyAsync(out_temb, p->temb, static_cast<size_t>(p->Bt) * ctx->D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int tpdm_tpm_forward(tpdm_plan* p, const float* x_nchw, const float* temb, float* out_alpha_beta, void* stream) {
  TPDM_CHECK(p && x_nchw && temb && out_alpha_beta, TPDM_ERR_ARG, "tpdm_tpm_forward: null argument");
  TPDM_CHECK(p->ctx->has_tpm, TPDM_ERR_STATE, "tpdm_tpm_forward: TimePredictor weights were not set");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  TPDM_TRY(k_nchw_to_nhwc_bf16(x_nchw, p->tpm_x, p->Bt, 2 * p->ctx->D, p->g, s));
  return run_tpm(p, p->Bt, temb, out_alpha_beta, s);
}

int tpdm_euler_step(const float* model_output, const float* sigma_next, const float* sigma, const float* sample, float* prev_sample,
                    int batch, long long n, void* stream) {
  TPDM_CHECK(model_output && sigma_next && sigma && sample && prev_sample, TPDM_ERR_ARG, "tpdm_euler_step: null argument");
  TPDM_CHECK(batch > 0 && n > 0, TPDM_ERR_SHAPE, "tpdm_euler_step: empty input");
  return k_euler(model_output, sigma_next, sigma, sample, prev_sample, batch, n, static_cast<cudaStream_t>(stream));
}

int tpdm_sample_begin(tpdm_plan* p, const float* latents, const float* neg_embeds, const float* pos_embeds, const float* neg_pooled,
                      const float* pos_pooled, float guidance_scale, int predict, const float* ratios, unsigned long long seed,
                      void* stream) {
  TPDM_CHECK(p && latents && neg_embeds && pos_embeds && neg_pooled && pos_pooled, TPDM_ERR_ARG, "tpdm_sample_begin: null argument");
  TPDM_CHECK(p->cfg_pairs, TPDM_ERR_STATE, "tpdm_sample_begin: the plan was created without cfg_pairs");
  TPDM_TRY(check_mode(p, in(Mode::kIdle) | in(Mode::kSample) | in(Mode::kQueue), "tpdm_sample_begin"));
  TPDM_CHECK(p->ctx->has_mmdit && p->ctx->has_tpm, TPDM_ERR_STATE, "tpdm_sample_begin: needs both MMDiT and TimePredictor weights");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  const size_t lat = static_cast<size_t>(p->B) * ctx->cfg.in_channels * p->Hl * p->Wl;
  p->predict = predict ? 1 : 0;
  p->have_ratios = ratios ? 1 : 0;
  p->seed = seed;
  TPDM_TRY(k_fill_f32(p->row_guidance, p->B, guidance_scale, s));
  TPDM_CUDA_OK(cudaMemcpyAsync(p->latents, latents, lat * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (ratios)
    TPDM_CUDA_OK(cudaMemcpyAsync(p->ratios, ratios, static_cast<size_t>(p->B) * p->max_steps * sizeof(float), cudaMemcpyDeviceToDevice, s));
  // sigma = ones (modeling_sd3_pnt.py:508); stream-ordered like everything else (no host staging, no synchronisation)
  TPDM_TRY(k_sample_init(p->sigma_hist, p->masks, p->all_done, p->B, p->max_steps, s));
  TPDM_TRY(set_prompts(p, neg_embeds, pos_embeds, neg_pooled, pos_pooled, s));
  p->mode = Mode::kSample;
  return 0;
}

int tpdm_sample_step(tpdm_plan* p, int step, void* stream) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_sample_step: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kSample), "tpdm_sample_step"));
  TPDM_CHECK(step >= 0 && step < p->max_steps, TPDM_ERR_ARG, "tpdm_sample_step: step %d outside [0,%d)", step, p->max_steps);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  const int D = ctx->D, B = p->B, T1 = p->max_steps + 1;
  const size_t lat = static_cast<size_t>(B) * ctx->cfg.in_channels * p->Hl * p->Wl;
  // a step enqueued after the batch finished (all_done[step-1] set, modeling_sd3_pnt.py:608) turns into empty launches
  set_skip_flag(step > 0 ? p->all_done + (step - 1) : nullptr);
  // timestep = sigma.repeat(2) * 1000 (modeling_sd3_pnt.py:526); latents duplicated inside patchify (:524)
  int st_mm = run_mmdit(p, p->latents, B, 2, p->sigma_hist + step, T1, 1000.0f, 2, nullptr, nullptr, true, s);
  set_skip_flag(nullptr);
  TPDM_TRY(st_mm);
  TPDM_TRY(k_cfg_combine(p->temb, p->temb_cfg, p->tembs + static_cast<size_t>(step) * B * D, B, D, p->row_guidance, s));
  TPDM_TRY(run_tpm(p, B, p->temb_cfg, p->alpha_beta, s));
  ScheduleArgs a;
  a.alpha_beta = p->alpha_beta;
  a.sigma_hist = p->sigma_hist;
  a.alphas = p->alphas;
  a.betas = p->betas;
  a.logprobs = p->logprobs;
  a.masks = p->masks;
  a.all_done = p->all_done;
  a.ratios = p->have_ratios ? p->ratios : nullptr;
  a.seed = p->seed;
  a.B = B;
  a.T = p->max_steps;
  a.step = step;
  a.predict = p->predict;
  a.relative = ctx->cfg.relative;
  a.prediction_type = ctx->cfg.prediction_type;
  a.min_sigma = ctx->cfg.min_sigma;
  a.epsilon = ctx->cfg.epsilon;
  TPDM_TRY(k_schedule(a, s));
  TPDM_TRY(k_unpatchify(p->pout, B, 1, p->row_guidance, ctx->cfg.out_channels, p->Hl, p->Wl, p->velocity, p->latents, p->sigma_hist + step,
                        p->sigma_hist + step + 1, T1, p->history + static_cast<size_t>(step) * lat, s));
  return 0;
}

int tpdm_sample_step_graph(tpdm_plan* p, int step, void* stream) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_sample_step_graph: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kSample), "tpdm_sample_step_graph"));
  TPDM_CHECK(step >= 0 && step < p->max_steps, TPDM_ERR_ARG, "tpdm_sample_step_graph: step %d outside [0,%d)", step, p->max_steps);
  // The Philox seed of a sampled trajectory is a kernel argument that changes with every call, and per-launch profiling records
  // events on the stream: both take the plain path.  (predict / injected ratios never read the seed.)
  if ((!p->predict && !p->have_ratios) || profiling_active()) return tpdm_sample_step(p, step, stream);
  if (p->graph_predict != p->predict || p->graph_have_ratios != p->have_ratios) {
    p->step_graph.clear();
    p->graph_predict = p->predict;
    p->graph_have_ratios = p->have_ratios;
  }
  if (p->step_graph.empty()) p->step_graph = std::vector<StepGraph>(p->max_steps);
  return replay_or_capture(p->step_graph[step], static_cast<cudaStream_t>(stream), "tpdm_sample_step_graph",
                           [&](cudaStream_t s) { return tpdm_sample_step(p, step, s); });
}

int tpdm_sample_state_get(tpdm_plan* p, tpdm_sample_state* out) {
  TPDM_CHECK(p && out, TPDM_ERR_ARG, "tpdm_sample_state_get: null argument");
  out->latents = p->latents;
  out->velocity = p->velocity;
  out->sigma_hist = p->sigma_hist;
  out->alphas = p->alphas;
  out->betas = p->betas;
  out->logprobs = p->logprobs;
  out->prob_masks = p->masks;
  out->all_done = p->all_done;
  out->tembs = p->tembs;
  out->tpm_input = p->tpm_x;
  out->history_latents = p->history;
  return 0;
}

// ---- device-side prompt queue ------------------------------------------------------------------------------------
namespace {
// text branch of every prompt + slot state + counters, in the order tpdm_queue_begin hands them out
void carve_queue(tpdm_plan* p, int n_prompts, Carver& c) {
  tpdm_plan::Queue& q = p->q;
  const size_t n = n_prompts, B = p->B, D = p->ctx->D;
  q.ctx0_all = c.take<float>(n * 2 * p->T * D);
  q.text_all = c.take<float>(n * 2 * D);
  q.sigma_cur = c.take<float>(2 * B);
  q.sigma_next = q.sigma_cur ? q.sigma_cur + B : nullptr;
  q.slot_prompt = c.take<int>(5 * B + 8);
  if (q.slot_prompt) {
    q.slot_step = q.slot_prompt + B;
    q.slot_flush = q.slot_step + B;
    q.slot_load = q.slot_flush + B;
    q.slot_active = q.slot_load + B;
    q.active = q.slot_active + B;
    q.idle_flag = q.active + 1;
  }
}
QueueArgs queue_args(const tpdm_plan* p, int init) {
  const tpdm_plan::Queue& q = p->q;
  QueueArgs a{};
  a.alpha_beta = p->alpha_beta;
  a.sigma_cur = q.sigma_cur;
  a.sigma_next = q.sigma_next;
  a.slot_prompt = q.slot_prompt;
  a.slot_step = q.slot_step;
  a.slot_flush = q.slot_flush;
  a.slot_load = q.slot_load;
  a.slot_active = q.slot_active;
  a.ticket = q.ticket;
  a.out_steps = q.out_steps;
  a.out_sigmas = q.out_sigmas;
  a.active = q.active;
  a.idle_flag = q.idle_flag;
  a.order = q.order;
  a.init_sigma = q.init_sigma;
  a.init_step = q.init_step;
  a.B = p->B;
  a.n_prompts = q.n_queued;
  a.max_steps = p->max_steps;
  a.relative = p->ctx->cfg.relative;
  a.prediction_type = p->ctx->cfg.prediction_type;
  a.init = init;
  a.min_sigma = p->ctx->cfg.min_sigma;
  a.epsilon = p->ctx->cfg.epsilon;
  a.predict = q.predict;
  a.seed = q.seed;
  a.ratios_all = q.ratios_all;
  a.rec_alphas = q.rec_alphas;
  a.rec_betas = q.rec_betas;
  a.rec_logprobs = q.rec_logprobs;
  a.row_guidance = p->row_guidance;
  if (p->mode == Mode::kStream) {
    const tpdm_plan::Stream& st = p->st;
    a.order = st.order;
    a.counters = st.counters;
    a.done_log = st.done_log;
    a.capacity = st.capacity;
    a.entry_guidance = st.guidance_all;
    a.entry_max_steps = st.max_steps_all;
    a.entry_predict = st.predict_all;
    a.entry_seed = st.seed_all;
    a.rec_alphas = st.rec_alphas;
    a.rec_betas = st.rec_betas;
    a.rec_logprobs = st.rec_logprobs;
  }
  return a;
}
int queue_move(tpdm_plan* p, cudaStream_t s) {
  const tpdm_plan::Queue& q = p->q;
  const long long lat = static_cast<long long>(p->ctx->cfg.in_channels) * p->Hl * p->Wl, ctx = static_cast<long long>(p->T) * p->ctx->D;
  return k_queue_move(q.slot_prompt, q.slot_flush, q.slot_load, p->B, lat, ctx, p->ctx->D, p->latents, q.noise_all, q.out_latents, p->ctx0,
                      q.ctx0_all, p->text_part, q.text_all, s);
}
}  // namespace

size_t tpdm_queue_workspace_bytes(const tpdm_plan* p, int n_prompts) {
  if (!p || n_prompts <= 0) return 0;
  tpdm_plan probe;
  probe.ctx = p->ctx;
  set_shape(&probe, p->B, p->cfg_pairs, p->Hl, p->Wl, p->T, p->max_steps);
  Carver c(nullptr);
  carve_queue(&probe, n_prompts, c);
  return c.off + 1024;
}

int tpdm_queue_begin(tpdm_plan* p, int n_prompts, const float* latents_all, const float* neg_embeds_all, const float* pos_embeds_all,
                     const float* neg_pooled_all, const float* pos_pooled_all, float guidance_scale, void* queue_workspace,
                     size_t queue_workspace_bytes, int* ticket, float* out_latents, int* out_steps, float* out_sigmas, const int* order,
                     int n_queued, const float* init_sigma, int init_step, void* stream) {
  TPDM_CHECK(p && latents_all && neg_embeds_all && pos_embeds_all && neg_pooled_all && pos_pooled_all && queue_workspace && ticket &&
                 out_latents && out_steps,
             TPDM_ERR_ARG, "tpdm_queue_begin: null argument");
  TPDM_CHECK(p->cfg_pairs, TPDM_ERR_STATE, "tpdm_queue_begin: the plan was created without cfg_pairs");
  TPDM_TRY(check_mode(p, in(Mode::kIdle) | in(Mode::kSample) | in(Mode::kQueue), "tpdm_queue_begin"));
  TPDM_CHECK(p->ctx->has_mmdit && p->ctx->has_tpm, TPDM_ERR_STATE, "tpdm_queue_begin: needs both MMDiT and TimePredictor weights");
  TPDM_CHECK(n_prompts >= p->B, TPDM_ERR_ARG, "tpdm_queue_begin: %d prompts for %d slots (use a plan with fewer slots)", n_prompts, p->B);
  TPDM_CHECK(order != nullptr || n_queued == n_prompts || n_queued <= 0, TPDM_ERR_ARG, "tpdm_queue_begin: n_queued needs an order table");
  TPDM_CHECK(n_queued <= n_prompts, TPDM_ERR_ARG, "tpdm_queue_begin: n_queued %d exceeds the %d prompts", n_queued, n_prompts);
  TPDM_CHECK(init_step >= 0 && init_step < p->max_steps && (init_step == 0) == (init_sigma == nullptr), TPDM_ERR_ARG,
             "tpdm_queue_begin: init_sigma and init_step (%d) go together, init_step < max_steps", init_step);
  const size_t need = tpdm_queue_workspace_bytes(p, n_prompts);
  TPDM_CHECK((reinterpret_cast<uintptr_t>(queue_workspace) & 1023) == 0 && queue_workspace_bytes >= need, TPDM_ERR_ARG,
             "tpdm_queue_begin: queue workspace must be 1 KiB aligned and >= %zu bytes", need);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  const int B = p->B, D = ctx->D, T = p->T, J = ctx->cfg.joint_attention_dim, PD = ctx->cfg.pooled_projection_dim;
  const size_t nctx = static_cast<size_t>(T) * D;
  tpdm_plan::Queue& q = p->q;
  q = tpdm_plan::Queue{};
  Carver c(queue_workspace);
  carve_queue(p, n_prompts, c);
  q.n_prompts = n_prompts;
  q.n_queued = n_queued > 0 ? n_queued : n_prompts;
  q.order = order;
  q.init_sigma = init_sigma;
  q.init_step = init_step;
  q.noise_all = latents_all;
  q.ticket = ticket;
  q.out_latents = out_latents;
  q.out_steps = out_steps;
  q.out_sigmas = out_sigmas;
  p->predict = 1;
  TPDM_TRY(k_fill_f32(p->row_guidance, B, guidance_scale, s));
  // sigma-independent text branch of every prompt, B prompts at a time through the plan's own buffers
  // (context_embedder + pooled-text MLP: transformer_sd3.py:337 and half of :336), parked per prompt as (uncond, cond)
  for (int c0 = 0; c0 < n_prompts; c0 += B) {
    const int start = c0 + B <= n_prompts ? c0 : n_prompts - B;  // the last chunk overlaps the previous one
    TPDM_TRY(set_prompts(p, neg_embeds_all + static_cast<size_t>(start) * T * J, pos_embeds_all + static_cast<size_t>(start) * T * J,
                         neg_pooled_all + static_cast<size_t>(start) * PD, pos_pooled_all + static_cast<size_t>(start) * PD, s));
    for (int b = 0; b < B; ++b)
      for (int half = 0; half < 2; ++half) {
        const size_t src = static_cast<size_t>(half) * B + b, dst = static_cast<size_t>(start + b) * 2 + half;
        TPDM_CUDA_OK(cudaMemcpyAsync(q.ctx0_all + dst * nctx, p->ctx0 + src * nctx, nctx * sizeof(float), cudaMemcpyDeviceToDevice, s));
        TPDM_CUDA_OK(cudaMemcpyAsync(q.text_all + dst * D, p->text_part + src * D, D * sizeof(float), cudaMemcpyDeviceToDevice, s));
      }
  }
  TPDM_CUDA_OK(cudaMemsetAsync(q.slot_prompt, 0xff, sizeof(int) * B, s));  // -1: every slot is idle and asks for a ticket
  TPDM_CUDA_OK(cudaMemsetAsync(q.slot_step, 0, sizeof(int) * (4 * B + 8), s));
  TPDM_TRY(k_queue_advance(queue_args(p, 1), s));
  TPDM_TRY(queue_move(p, s));
  p->mode = Mode::kQueue;
  return 0;
}

int tpdm_queue_step(tpdm_plan* p, void* stream) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_queue_step: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kQueue) | in(Mode::kStream), "tpdm_queue_step"));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  const int B = p->B;
  // a step enqueued after the queue drained (idle_flag set) turns into empty launches
  set_skip_flag(p->q.idle_flag);
  // emptied slots (the tail of the queue) are skipped tile by tile / CTA by CTA inside the heavy kernels
  if (B > 1) set_batch_mask(p->q.slot_active, B);
  int st_mm = run_mmdit(p, p->latents, B, 2, p->q.sigma_cur, 1, 1000.0f, 2, nullptr, nullptr, true, s);
  set_skip_flag(nullptr);
  if (st_mm == 0) st_mm = k_cfg_combine(p->temb, p->temb_cfg, nullptr, B, ctx->D, p->row_guidance, s);
  if (st_mm == 0) st_mm = run_tpm(p, B, p->temb_cfg, p->alpha_beta, s);
  set_batch_mask(nullptr, 1);
  TPDM_TRY(st_mm);
  const tpdm_plan::Queue& q = p->q;
  if (q.rec_tembs || q.rec_tpm)  // before queue_advance moves the slots on
    TPDM_TRY(k_queue_record(q.slot_prompt, q.slot_step, B, p->max_steps, ctx->D, p->temb_cfg, q.rec_tembs, p->tpm_x, q.rec_tpm,
                            static_cast<long long>(p->g) * p->g * 2 * ctx->D, s));
  TPDM_TRY(k_queue_schedule(queue_args(p, 0), s));
  TPDM_TRY(k_unpatchify(p->pout, B, 1, p->row_guidance, ctx->cfg.out_channels, p->Hl, p->Wl, nullptr, p->latents, p->q.sigma_cur,
                        p->q.sigma_next, 1, nullptr, s));
  TPDM_TRY(p->mode == Mode::kStream ? k_stream_advance(queue_args(p, 0), 0, s) : k_queue_advance(queue_args(p, 0), s));
  TPDM_TRY(queue_move(p, s));
  return 0;
}

int tpdm_queue_set_rollout(tpdm_plan* p, unsigned long long seed, const float* ratios_all, float* alphas, float* betas, float* logprobs,
                           float* tembs, void* tpm_inputs) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_queue_set_rollout: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kQueue), "tpdm_queue_set_rollout"));  // a prompt stream takes the mode per request
  // the probe step of longest-first scheduling ran the Beta mode, so such a queue cannot start sampled trajectories
  TPDM_CHECK(p->q.init_step == 0, TPDM_ERR_STATE, "tpdm_queue_set_rollout: the queue began after %d probe steps (init_step > 0)", p->q.init_step);
  tpdm_plan::Queue& q = p->q;
  q.graph.drop();  // the captured step holds the predict-mode arguments
  q.predict = 0;
  q.seed = seed;
  q.ratios_all = ratios_all;
  q.rec_alphas = alphas;
  q.rec_betas = betas;
  q.rec_logprobs = logprobs;
  q.rec_tembs = tembs;
  q.rec_tpm = static_cast<bf16*>(tpm_inputs);
  return 0;
}

int tpdm_queue_step_graph(tpdm_plan* p, void* stream) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_queue_step_graph: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kQueue) | in(Mode::kStream), "tpdm_queue_step_graph"));
  // a queue step has no host-side argument that changes between steps (a rollout's seed is fixed for the whole drain):
  // capture it once, replay it every step
  return replay_or_capture(p->q.graph, static_cast<cudaStream_t>(stream), "tpdm_queue_step_graph",
                           [&](cudaStream_t s) { return tpdm_queue_step(p, s); });
}

int tpdm_queue_status(tpdm_plan* p, const int** active_slots, const int** slot_prompts) {
  TPDM_CHECK(p, TPDM_ERR_STATE, "tpdm_queue_status: call tpdm_queue_begin first");
  TPDM_TRY(check_mode(p, in(Mode::kQueue) | in(Mode::kStream), "tpdm_queue_status"));
  if (active_slots) *active_slots = p->q.active;
  if (slot_prompts) *slot_prompts = p->q.slot_prompt;
  return 0;
}

// ---- open prompt stream -------------------------------------------------------------------------------------------
namespace {
// ring of `capacity` entries + slot state + counters + admission staging, in the order tpdm_stream_open hands them out
void carve_stream(tpdm_plan* p, int capacity, Carver& c) {
  tpdm_plan::Queue& q = p->q;
  tpdm_plan::Stream& st = p->st;
  const size_t cap = capacity, B = p->B, T = p->T, D = p->ctx->D, J = p->ctx->cfg.joint_attention_dim;
  const size_t lat = static_cast<size_t>(p->ctx->cfg.in_channels) * p->Hl * p->Wl;
  st.noise = c.take<float>(cap * lat);
  q.ctx0_all = c.take<float>(cap * 2 * T * D);
  q.text_all = c.take<float>(cap * 2 * D);
  q.out_latents = c.take<float>(cap * lat);
  q.out_sigmas = c.take<float>(cap * (p->max_steps + 1));
  q.out_steps = c.take<int>(cap);
  st.order = c.take<int>(cap);
  st.done_log = c.take<int>(cap);
  st.guidance_all = c.take<float>(cap);
  st.max_steps_all = c.take<int>(cap);
  st.predict_all = c.take<int>(cap);
  st.seed_all = c.take<unsigned long long>(cap);
  st.rec_alphas = c.take<float>(cap * p->max_steps);
  st.rec_betas = c.take<float>(cap * p->max_steps);
  st.rec_logprobs = c.take<float>(cap * p->max_steps);
  q.sigma_cur = c.take<float>(2 * B);
  q.sigma_next = q.sigma_cur ? q.sigma_cur + B : nullptr;
  q.slot_prompt = c.take<int>(5 * B + kStreamCounters + 2);
  if (q.slot_prompt) {
    q.slot_step = q.slot_prompt + B;
    q.slot_flush = q.slot_step + B;
    q.slot_load = q.slot_flush + B;
    q.slot_active = q.slot_load + B;
    st.counters = q.slot_active + B;
    q.active = st.counters + kStreamCounters;   // right behind the counters: one copy reads both
    q.idle_flag = q.active + 1;
  }
  st.enc = c.take<bf16>(2 * B * T * J);
  st.ctx0 = c.take<float>(2 * B * T * D);
  st.phid = c.take<float>(2 * B * D);
  st.text = c.take<float>(2 * B * D);
}

// context_embedder + pooled-text MLP of n <= slots prompts into the staging rows 2k + half (half 0 = negative, 1 = positive)
int stream_embed(tpdm_plan* p, int n, const float* neg, const float* pos, const float* neg_pooled, const float* pos_pooled, cudaStream_t s) {
  const tpdm_ctx* ctx = p->ctx;
  const tpdm_weights& w = ctx->w;
  tpdm_plan::Stream& st = p->st;
  const int D = ctx->D, PD = ctx->cfg.pooled_projection_dim;
  const long long row = static_cast<long long>(p->T) * ctx->cfg.joint_attention_dim;
  for (int k = 0; k < n; ++k) {
    TPDM_TRY(k_cast_bf16(neg + k * row, st.enc + (2 * k) * row, row, s));
    TPDM_TRY(k_cast_bf16(pos + k * row, st.enc + (2 * k + 1) * row, row, s));
  }
  GemmOp op = st.ctx_embed;   // the TMA maps cover 2 * slots rows; run the first 2n
  op.batch = 2 * n;
  op.num_tiles = op.batch * op.tiles_m_per_batch * op.tiles_n;
  TPDM_TRY(gemm_launch(&op, 1, s));
  TPDM_TRY(k_gemv_f32(w.p_w1, w.p_b1, neg_pooled, PD, nullptr, st.phid, 2 * D, n, D, PD, 0, s));
  TPDM_TRY(k_gemv_f32(w.p_w1, w.p_b1, pos_pooled, PD, nullptr, st.phid + D, 2 * D, n, D, PD, 0, s));
  TPDM_TRY(k_gemv_f32(w.p_w2, w.p_b2, st.phid, D, nullptr, st.text, D, 2 * n, D, D, 1, s));
  return 0;
}
}  // namespace

size_t tpdm_stream_workspace_bytes(const tpdm_plan* p, int capacity) {
  if (!p || capacity <= 0) return 0;
  tpdm_plan probe;
  probe.ctx = p->ctx;
  set_shape(&probe, p->B, p->cfg_pairs, p->Hl, p->Wl, p->T, p->max_steps);
  Carver c(nullptr);
  carve_stream(&probe, capacity, c);
  return c.off + 1024;
}

int tpdm_stream_open(tpdm_plan* p, int capacity, float guidance_scale, void* workspace, size_t workspace_bytes, void* stream) {
  TPDM_CHECK(p && workspace, TPDM_ERR_ARG, "tpdm_stream_open: null argument");
  TPDM_CHECK(p->cfg_pairs, TPDM_ERR_STATE, "tpdm_stream_open: the plan was created without cfg_pairs");
  TPDM_CHECK(p->ctx->has_mmdit && p->ctx->has_tpm, TPDM_ERR_STATE, "tpdm_stream_open: needs both MMDiT and TimePredictor weights");
  TPDM_TRY(check_mode(p, in(Mode::kIdle) | in(Mode::kSample), "tpdm_stream_open"));
  TPDM_CHECK(capacity > 0, TPDM_ERR_ARG, "tpdm_stream_open: capacity %d must be positive", capacity);
  const size_t need = tpdm_stream_workspace_bytes(p, capacity);
  TPDM_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0 && workspace_bytes >= need, TPDM_ERR_ARG,
             "tpdm_stream_open: workspace must be 1 KiB aligned and >= %zu bytes", need);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  const int B = p->B, T = p->T, D = ctx->D, J = ctx->cfg.joint_attention_dim;
  tpdm_plan::Queue& q = p->q;
  tpdm_plan::Stream& st = p->st;
  q = tpdm_plan::Queue{};
  Carver c(workspace);
  carve_stream(p, capacity, c);
  TPDM_TRY(gemm_op_init(&st.ctx_embed, st.enc, J, static_cast<long long>(T) * J, T, 2 * B, J, ctx->w.ctx_w, D, EPI_BIAS_F32, st.ctx0,
                        static_cast<long long>(T) * D, D, ctx->w.ctx_b, nullptr, 0));
  st.capacity = capacity;
  st.guidance = guidance_scale;
  q.n_prompts = q.n_queued = capacity;
  q.noise_all = st.noise;
  p->predict = 1;
  TPDM_TRY(k_fill_f32(p->row_guidance, B, guidance_scale, s));   // idle rows; a slot takes its request's value when it claims one
  TPDM_CUDA_OK(cudaMemsetAsync(q.sigma_cur, 0, sizeof(float) * 2 * B, s));
  TPDM_CUDA_OK(cudaMemsetAsync(q.slot_prompt, 0xff, sizeof(int) * B, s));  // -1: every slot is idle
  TPDM_CUDA_OK(cudaMemsetAsync(q.slot_step, 0, sizeof(int) * (4 * B + kStreamCounters + 2), s));
  p->mode = Mode::kStream;
  TPDM_TRY(k_stream_advance(queue_args(p, 0), 1, s));   // nothing submitted: every slot stays idle, the skip flag is raised
  return 0;
}

int tpdm_stream_submit_options(tpdm_plan* p, int n, const int* entry_ids, const float* latents, const float* neg_embeds,
                               const float* pos_embeds, const float* neg_pooled, const float* pos_pooled, const tpdm_request_options* options,
                               void* stream) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_stream_submit: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kStream), "tpdm_stream_submit"));
  TPDM_CHECK(n > 0 && entry_ids && latents && neg_embeds && pos_embeds && neg_pooled && pos_pooled, TPDM_ERR_ARG,
             "tpdm_stream_submit: null argument or n <= 0");
  tpdm_plan::Stream& st = p->st;
  TPDM_CHECK(n <= st.capacity, TPDM_ERR_ARG, "tpdm_stream_submit: %d prompts for a ring of %d entries", n, st.capacity);
  std::vector<char> seen(st.capacity, 0);   // a repeated id would publish one entry twice and overrun unclaimed order slots
  for (int k = 0; k < n; ++k) {
    const int id = entry_ids[k];
    TPDM_CHECK(id >= 0 && id < st.capacity, TPDM_ERR_ARG, "tpdm_stream_submit: entry id %d outside [0,%d)", id, st.capacity);
    TPDM_CHECK(!seen[id], TPDM_ERR_ARG, "tpdm_stream_submit: entry id %d given twice", id);
    seen[id] = 1;
  }
  for (int k = 0; options && k < n; ++k) {
    const tpdm_request_options& o = options[k];
    TPDM_CHECK(std::isfinite(o.guidance_scale), TPDM_ERR_ARG, "tpdm_stream_submit: prompt %d: guidance_scale is not finite", k);
    TPDM_CHECK(o.max_steps >= 1 && o.max_steps <= p->max_steps, TPDM_ERR_ARG, "tpdm_stream_submit: prompt %d: max_steps %d outside [1,%d]", k,
               o.max_steps, p->max_steps);
    TPDM_CHECK(o.predict == 0 || o.predict == 1, TPDM_ERR_ARG, "tpdm_stream_submit: prompt %d: predict %d is neither 0 nor 1", k, o.predict);
    TPDM_CHECK(o.reserved == 0, TPDM_ERR_ARG, "tpdm_stream_submit: prompt %d: reserved is %d, must be 0", k, o.reserved);
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const tpdm_ctx* ctx = p->ctx;
  tpdm_plan::Queue& q = p->q;
  const int D = ctx->D, PD = ctx->cfg.pooled_projection_dim;
  const size_t nctx = static_cast<size_t>(p->T) * D, row = static_cast<size_t>(p->T) * ctx->cfg.joint_attention_dim;
  const size_t lat = static_cast<size_t>(ctx->cfg.in_channels) * p->Hl * p->Wl;
  const int pass = p->B < kStreamPublishMax ? p->B : kStreamPublishMax;
  const tpdm_request_options defaults{st.guidance, p->max_steps, 1, 0, 0};
  for (int k0 = 0; k0 < n; k0 += pass) {
    const int m = n - k0 < pass ? n - k0 : pass;
    TPDM_TRY(stream_embed(p, m, neg_embeds + k0 * row, pos_embeds + k0 * row, neg_pooled + static_cast<size_t>(k0) * PD,
                          pos_pooled + static_cast<size_t>(k0) * PD, s));
    StreamEntries e{};
    for (int k = 0; k < m; ++k) {
      const size_t id = entry_ids[k0 + k];
      const tpdm_request_options& o = options ? options[k0 + k] : defaults;
      e.id[k] = static_cast<int>(id);
      e.guidance[k] = o.guidance_scale;
      e.max_steps[k] = o.max_steps;
      e.predict[k] = o.predict;
      e.seed[k] = o.seed;
      TPDM_CUDA_OK(cudaMemcpyAsync(st.noise + id * lat, latents + (k0 + k) * lat, lat * sizeof(float), cudaMemcpyDeviceToDevice, s));
      TPDM_CUDA_OK(cudaMemcpyAsync(q.ctx0_all + id * 2 * nctx, st.ctx0 + static_cast<size_t>(k) * 2 * nctx, 2 * nctx * sizeof(float),
                                   cudaMemcpyDeviceToDevice, s));
      TPDM_CUDA_OK(cudaMemcpyAsync(q.text_all + id * 2 * D, st.text + static_cast<size_t>(k) * 2 * D, 2 * D * sizeof(float),
                                   cudaMemcpyDeviceToDevice, s));
    }
    TPDM_TRY(k_stream_publish(queue_args(p, 0), st.order, e, m, s));
  }
  // idle slots take the new tickets now, so the next step already computes them
  TPDM_TRY(k_stream_advance(queue_args(p, 0), 1, s));
  return queue_move(p, s);
}

int tpdm_stream_submit(tpdm_plan* p, int n, const int* entry_ids, const float* latents, const float* neg_embeds, const float* pos_embeds,
                       const float* neg_pooled, const float* pos_pooled, void* stream) {
  return tpdm_stream_submit_options(p, n, entry_ids, latents, neg_embeds, pos_embeds, neg_pooled, pos_pooled, nullptr, stream);
}

int tpdm_stream_records(tpdm_plan* p, const float** alphas, const float** betas, const float** logprobs) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_stream_records: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kStream), "tpdm_stream_records"));
  if (alphas) *alphas = p->st.rec_alphas;
  if (betas) *betas = p->st.rec_betas;
  if (logprobs) *logprobs = p->st.rec_logprobs;
  return 0;
}

int tpdm_stream_status(tpdm_plan* p, const int** counters, const int** done_log, const float** out_latents, const int** out_steps,
                       const float** out_sigmas) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_stream_status: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kStream), "tpdm_stream_status"));
  if (counters) *counters = p->st.counters;
  if (done_log) *done_log = p->st.done_log;
  if (out_latents) *out_latents = p->q.out_latents;
  if (out_steps) *out_steps = p->q.out_steps;
  if (out_sigmas) *out_sigmas = p->q.out_sigmas;
  return 0;
}

int tpdm_stream_close(tpdm_plan* p) {
  TPDM_CHECK(p, TPDM_ERR_ARG, "tpdm_stream_close: null plan");
  TPDM_TRY(check_mode(p, in(Mode::kStream), "tpdm_stream_close"));
  p->st = tpdm_plan::Stream{};
  p->q = tpdm_plan::Queue{};
  p->mode = Mode::kIdle;
  return 0;
}

// ---- unit entry points ----------------------------------------------------------------------------------------
int tpdm_gemm_bf16(const void* A, const void* W, const float* bias, const float* gate, void* out, int batch, int rows, int N, int K, int epi,
                   void* stream) {
  TPDM_CHECK(A && W && out, TPDM_ERR_ARG, "tpdm_gemm_bf16: null argument");
  TPDM_CHECK(epi >= 0 && epi <= 3, TPDM_ERR_ARG, "tpdm_gemm_bf16: epilogue %d unknown", epi);
  GemmOp op;
  TPDM_TRY(gemm_op_init(&op, A, K, static_cast<long long>(rows) * K, rows, batch, K, W, N, epi, out, static_cast<long long>(rows) * N, N, bias,
                        gate, N));
  return gemm_launch(&op, 1, static_cast<cudaStream_t>(stream));
}

int tpdm_joint_attention(const void* qkv, void* out, int Bt, int S, int H, int dp, int head_dim, int q_rows, void* stream) {
  TPDM_CHECK(qkv && out, TPDM_ERR_ARG, "tpdm_joint_attention: null argument");
  AttnOp op;
  TPDM_TRY(attn_op_init(&op, qkv, Bt, S, H, dp, head_dim, out));
  if (q_rows > 0 && q_rows < S) op.q_tiles = (q_rows + 127) / 128;
  return attn_launch(&op, static_cast<cudaStream_t>(stream));
}

int tpdm_attention_redo_count(void) { return attn_redo_count(); }
long long tpdm_attention_redo_total(void) { return attn_redo_total(); }

int tpdm_conv3x3_nhwc(const void* x, const void* w, const float* bias, float* out, int batch, int g, int C, int N, void* stream) {
  TPDM_CHECK(x && w && out, TPDM_ERR_ARG, "tpdm_conv3x3_nhwc: null argument");
  GemmOp op;
  TPDM_TRY(gemm_op_init_conv3x3(&op, x, batch, g, C, w, N, EPI_BIAS_F32, out, N, bias));
  return gemm_launch(&op, 1, static_cast<cudaStream_t>(stream));
}

int tpdm_conv3x3_wgrad(const void* dyt, const void* x_shifted_nchw, float* dw, int samples, int g, int C, int M, void* stream) {
  TPDM_CHECK(dyt && x_shifted_nchw && dw, TPDM_ERR_ARG, "tpdm_conv3x3_wgrad: null argument");
  GemmOp op;
  TPDM_TRY(gemm_op_init_conv3x3_wgrad(&op, dyt, x_shifted_nchw, samples, g, C, M, dw));
  return gemm_launch(&op, 1, static_cast<cudaStream_t>(stream));
}

int tpdm_ln_modulate(const float* x, const float* shift, const float* scale, int mod_stride, void* out_bf16, int batch, int rows, int D,
                     void* stream) {
  TPDM_CHECK(x && shift && scale && out_bf16, TPDM_ERR_ARG, "tpdm_ln_modulate: null argument");
  LnSeg seg{x, reinterpret_cast<bf16*>(out_bf16), shift, scale, rows, batch, mod_stride};
  return k_ln_modulate(&seg, 1, D, static_cast<cudaStream_t>(stream));
}

int tpdm_ln_modulate_pair(const float* x0, const float* shift0, const float* scale0, void* out0_bf16, int rows0, const float* x1,
                          const float* shift1, const float* scale1, void* out1_bf16, int rows1, int mod_stride, int batch, int D,
                          void* stream) {
  TPDM_CHECK(x0 && shift0 && scale0 && out0_bf16 && x1 && shift1 && scale1 && out1_bf16, TPDM_ERR_ARG,
             "tpdm_ln_modulate_pair: null argument");
  TPDM_CHECK(rows0 > 0 && rows1 > 0 && batch > 0, TPDM_ERR_SHAPE, "tpdm_ln_modulate_pair: rows %d / %d, batch %d", rows0, rows1, batch);
  const LnSeg seg[2] = {LnSeg{x0, reinterpret_cast<bf16*>(out0_bf16), shift0, scale0, rows0, batch, mod_stride},
                        LnSeg{x1, reinterpret_cast<bf16*>(out1_bf16), shift1, scale1, rows1, batch, mod_stride}};
  return k_ln_modulate(seg, 2, D, static_cast<cudaStream_t>(stream));
}

int tpdm_quantize_fp8_rows(const float* x, int rows, int K, void* codes, float* scales, void* stream) {
  TPDM_CHECK(x && codes && scales, TPDM_ERR_ARG, "tpdm_quantize_fp8_rows: null argument");
  return k_quantize_fp8_rows(x, rows, K, static_cast<uint8_t*>(codes), scales, static_cast<cudaStream_t>(stream));
}

int tpdm_ln_modulate_fp8(const float* x, const float* shift, const float* scale, int mod_stride, void* out_codes, float* out_scales,
                         int batch, int rows, int D, void* stream) {
  TPDM_CHECK(x && shift && scale && out_codes && out_scales, TPDM_ERR_ARG, "tpdm_ln_modulate_fp8: null argument");
  LnSeg seg{x, nullptr, shift, scale, rows, batch, mod_stride, static_cast<uint8_t*>(out_codes), out_scales};
  return k_ln_modulate(&seg, 1, D, static_cast<cudaStream_t>(stream));
}

int tpdm_gemm_fp8(const void* A8, const float* a_scale, const void* W8, const float* w_scale, const float* bias, void* out, int batch,
                  int rows, int N, int K, int epi, void* stream) {
  TPDM_CHECK(A8 && a_scale && W8 && w_scale && out, TPDM_ERR_ARG, "tpdm_gemm_fp8: null argument");
  TPDM_CHECK(epi >= 0 && epi <= 2, TPDM_ERR_ARG, "tpdm_gemm_fp8: epilogue %d unknown", epi);
  GemmOp op;
  TPDM_TRY(gemm_op_init_fp8(&op, A8, K, static_cast<long long>(rows) * K, a_scale, rows, batch, K, W8, w_scale, N, epi, out,
                            static_cast<long long>(rows) * N, N, bias));
  return gemm_launch(&op, 1, static_cast<cudaStream_t>(stream));
}

int tpdm_set_launch_guards(const int* skip, const int* slot_active, int slots) {
  TPDM_CHECK(slots >= 1, TPDM_ERR_ARG, "tpdm_set_launch_guards: slots %d < 1", slots);
  set_skip_flag(skip);
  set_batch_mask(slot_active, slots);
  return 0;
}

int tpdm_gemm_ops(const tpdm_gemm_op_desc* ops, int n_ops, void* stream) {
  TPDM_CHECK(ops, TPDM_ERR_ARG, "tpdm_gemm_ops: null argument");
  TPDM_CHECK(n_ops >= 1 && n_ops <= 2, TPDM_ERR_ARG, "tpdm_gemm_ops: %d ops (1 or 2 per launch)", n_ops);
  for (int i = 0; i < n_ops; ++i) {
    const tpdm_gemm_op_desc& d = ops[i];
    TPDM_CHECK(d.A && d.W && d.out, TPDM_ERR_ARG, "tpdm_gemm_ops: op %d: null argument", i);
    TPDM_CHECK(d.epi >= 0 && d.epi <= 3, TPDM_ERR_ARG, "tpdm_gemm_ops: op %d: epilogue %d unknown", i, d.epi);
    TPDM_CHECK((d.a_scale == nullptr) == (d.w_scale == nullptr), TPDM_ERR_ARG, "tpdm_gemm_ops: op %d: E4M3 operands need both scales", i);
  }
  GemmOp g[2];
  for (int i = 0; i < n_ops; ++i) {
    const tpdm_gemm_op_desc& d = ops[i];
    if (d.a_scale)
      TPDM_TRY(gemm_op_init_fp8(&g[i], d.A, d.a_row_stride, d.a_batch_stride, d.a_scale, d.rows, d.batch, d.K, d.W, d.w_scale, d.N, d.epi,
                                d.out, d.out_batch_stride, d.ldo, d.bias));
    else
      TPDM_TRY(gemm_op_init(&g[i], d.A, d.a_row_stride, d.a_batch_stride, d.rows, d.batch, d.K, d.W, d.N, d.epi, d.out, d.out_batch_stride,
                            d.ldo, d.bias, d.gate, d.gate_stride));
    TPDM_TRY(gemm_op_set_ksplit(&g[i], d.ksplit));
  }
  return gemm_launch(g, n_ops, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
