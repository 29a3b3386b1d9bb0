"""Drop-in for /root/reference/src/models/stable_diffusion_3/modeling_sd3_pnt.py (the TPDM-wrapped SD3 pipeline).

Same class names, constructor kwargs, method names and output fields as the reference; the denoising loop
(modeling_sd3_pnt.py:522-612), the TimePredictor (:85-126) and the Euler update run in libtpdm_b200.so.
Out of scope (SURVEY.md section 8): the three text encoders and the VAE -- pass ``prompt_embeds`` etc.; ``images`` is
filled only when a ``vae`` module with ``decode`` has been attached by the caller.
"""
from __future__ import annotations

import json
import logging
import os
from typing import List, Optional, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from .engine import Engine
from .model_utilis import CustomDiffusionModelOutput, CustomFlowMatchEulerDiscreteScheduler
from .reference_distributions import get_ref_beta
from .transformer_sd3 import CustomSD3Transformer2DModel

logger = logging.getLogger(__name__)

SD3_MEDIUM_TRANSFORMER_CONFIG = dict(
    sample_size=128, patch_size=2, in_channels=16, num_layers=24, attention_head_dim=64, num_attention_heads=24,
    joint_attention_dim=4096, caption_projection_dim=1536, pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=192)


def _check_loaded(what: str, result, ignore_unexpected=()):
    """``load_state_dict(strict=False)`` must not silently leave random-init weights behind (from_pretrained reports them)."""
    missing = list(result.missing_keys)
    unexpected = [k for k in result.unexpected_keys if not k.startswith(tuple(ignore_unexpected))] if ignore_unexpected else list(result.unexpected_keys)
    if missing:
        raise ValueError(f"{what} checkpoint is missing {len(missing)} tensors, e.g. {missing[:4]}")
    if unexpected:
        logger.warning("%s checkpoint has %d tensors this module does not use, e.g. %s", what, len(unexpected), unexpected[:4])


def reshape_hidden_states_to_2d(hidden_states: torch.Tensor, height: int = 64, width: int = 64, patch_size: int = 2) -> torch.Tensor:
    """modeling_sd3_pnt.py:33-54 (a pure re-indexing; the CUDA path folds it into its store addresses instead)."""
    hidden_states = hidden_states.reshape(
        shape=(hidden_states.shape[0], height // patch_size, width // patch_size, patch_size, patch_size, hidden_states.shape[-1]))
    hidden_states = torch.einsum("nhwpqc->nchpwq", hidden_states)
    return hidden_states.reshape(shape=(hidden_states.shape[0], hidden_states.shape[1], height, width))


class CustomAdaGroupNormZeroSingle(nn.Module):
    """Parameter container with the reference's names (modeling_sd3_pnt.py:56-83): ``linear`` (D -> 2C), ``norm`` = GroupNorm(1, C)."""

    def __init__(self, input_dim: int, embedding_dim: int, norm_type="group_norm", bias=True, device=None, dtype=None):
        super().__init__()
        self.silu = nn.SiLU()
        self.linear = nn.Linear(input_dim, 2 * embedding_dim, bias=bias, device=device, dtype=dtype)
        if norm_type == "group_norm":
            self.norm = nn.GroupNorm(1, embedding_dim, eps=1e-6, device=device, dtype=dtype)
        else:
            raise ValueError(f"Unsupported `norm_type` ({norm_type}) provided. Supported ones are: 'layer_norm', 'fp32_layer_norm'.")


class TimePredictor(nn.Module):
    """modeling_sd3_pnt.py:85-126.  forward(x (B, in_channels, g, g), temb (B, in_channels/2)) -> (B, 2) = (alpha, beta) > 1."""

    def __init__(self, conv_out_channels, in_channels=1536 * 2, projection_dim=2, init_alpha=1.5, init_beta=0.5, device=None, dtype=None):
        super().__init__()
        if projection_dim != 2:
            raise ValueError("projection_dim must be 2 (alpha, beta)")
        fk = {"device": device, "dtype": dtype}
        self.conv1 = nn.Conv2d(in_channels, conv_out_channels, kernel_size=(3, 3), padding=1, **fk)
        self.conv2 = nn.Conv2d(conv_out_channels, conv_out_channels, kernel_size=(3, 3), padding=1, stride=2, **fk)
        self.fc1 = nn.Linear(conv_out_channels, 128, **fk)
        self.fc2 = nn.Linear(128, projection_dim, **fk)
        self.norm1 = CustomAdaGroupNormZeroSingle(in_channels // 2, conv_out_channels, **fk)
        self.epsilon = 1.0
        self.init_alpha = init_alpha
        self.init_beta = init_beta
        self.in_channels, self.conv_out_channels = in_channels, conv_out_channels
        self._init_weights()
        self._engine: Optional[Engine] = None
        self._engine_key = None

    def _init_weights(self):
        for m in self.modules():
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                nn.init.normal_(m.weight, std=0.02)
                if m.bias is not None and isinstance(m, nn.Conv2d):
                    nn.init.constant_(m.bias, 0)
        nn.init.constant_(self.fc1.bias, 0)
        nn.init.constant_(self.fc2.bias[0], self.init_alpha)
        nn.init.constant_(self.fc2.bias[1], self.init_beta)

    def _weights_key(self):
        return tuple((p.data_ptr(), p._version, p.device) for p in self.parameters())

    def _standalone_engine(self) -> Engine:
        key = self._weights_key()
        if self._engine is None or key != self._engine_key:
            D = self.in_channels // 2
            if D % 64 != 0:
                raise ValueError("TimePredictor in_channels/2 must be a multiple of 64 for the CUDA path")
            cfg = dict(num_layers=1, num_attention_heads=D // 64, attention_head_dim=64, joint_attention_dim=4096,
                       pooled_projection_dim=2048, in_channels=16, out_channels=16, patch_size=2, pos_embed_max_size=192, qk_norm=None)
            self._engine = Engine(cfg, self.fc2.weight.device, tpm_sd=self.state_dict(), tpm_epsilon=self.epsilon,
                                  tpm_channels=self.conv_out_channels)
            self._engine_key = key
        return self._engine

    @torch.no_grad()
    def forward(self, x, temb):
        return self._standalone_engine().tpm_forward(x, temb).to(x.dtype)


class SD3PredictNextTimeStepModel(nn.Module):
    def __init__(
        self,
        pretrained_model_name_or_path=None,
        torch_dtype=torch.float16,
        min_sigma=0.001,
        init_alpha=1.5,
        init_beta=0.5,
        pre_process=False,
        relative=True,
        prediction_type="alpha_beta",
        transformer_config: Optional[dict] = None,
        device=None,
        vae_config: Optional[dict] = None,
        mmdit_precision: str = "bf16",
    ):
        """Reference kwargs (modeling_sd3_pnt.py:130-140) plus ``transformer_config`` / ``device`` for offline random-init
        construction (the reference only has ``from_pretrained``) and ``mmdit_precision`` ("bf16" or "fp8", see
        CustomSD3Transformer2DModel), which is the transformer's attribute of that name."""
        super().__init__()
        cfg = transformer_config
        weights_file = None
        if cfg is None:
            if pretrained_model_name_or_path is None:
                raise ValueError("give either pretrained_model_name_or_path or transformer_config")
            cfg_path = os.path.join(pretrained_model_name_or_path, "transformer", "config.json")
            if not os.path.isfile(cfg_path):
                raise ValueError(f"{cfg_path} not found (no network: only local diffusers-layout checkpoints can be loaded)")
            raw = json.load(open(cfg_path))
            cfg = {k: raw[k] for k in SD3_MEDIUM_TRANSFORMER_CONFIG if k in raw}
            for k in ("qk_norm", "dual_attention_layers"):
                if k in raw:
                    cfg[k] = raw[k]
            weights_file = os.path.join(pretrained_model_name_or_path, "transformer", "diffusion_pytorch_model.safetensors")
        # VAE (SURVEY 8(f) rank 1): built from `vae_config` or <path>/vae/config.json; otherwise None and the caller may attach
        # any module with .decode / .config.  Only the decoder exists (tpdm_b200/vae.py); images stay off when vae is None.
        self.vae = None
        vae_weights = None
        if vae_config is None and pretrained_model_name_or_path is not None:
            vcfg_path = os.path.join(pretrained_model_name_or_path, "vae", "config.json")
            if os.path.isfile(vcfg_path):
                rawv = json.load(open(vcfg_path))
                vae_config = {k: rawv[k] for k in ("latent_channels", "out_channels", "block_out_channels", "layers_per_block",
                                                   "norm_num_groups", "scaling_factor", "shift_factor") if k in rawv}
                vae_weights = os.path.join(pretrained_model_name_or_path, "vae", "diffusion_pytorch_model.safetensors")
        if vae_config is not None:
            from .vae import AutoencoderKL

            self.vae = AutoencoderKL(**vae_config, device=device, dtype=torch_dtype)
            if vae_weights is not None and os.path.isfile(vae_weights):
                from safetensors.torch import load_file

                _check_loaded("vae", self.vae.load_state_dict(load_file(vae_weights), strict=False), ("encoder.", "quant_conv.", "post_quant_conv."))
        self.transformer = CustomSD3Transformer2DModel(**cfg, device=device, dtype=torch_dtype, mmdit_precision=mmdit_precision)
        if weights_file is not None and os.path.isfile(weights_file):
            from safetensors.torch import load_file

            _check_loaded("transformer", self.transformer.load_state_dict(load_file(weights_file), strict=False))
        self.time_predictor = TimePredictor(
            conv_out_channels=128, in_channels=self.transformer.config.caption_projection_dim * 2, projection_dim=2,
            init_alpha=init_alpha, init_beta=init_beta, device=device, dtype=torch_dtype)
        self.scheduler = CustomFlowMatchEulerDiscreteScheduler()
        self.pre_process = pre_process
        self.vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1) if self.vae is not None else 8   # :181-183
        self.tokenizer_max_length = 77
        self.default_sample_size = self.transformer.config.sample_size
        self.patch_size = self.transformer.config.patch_size
        self.min_sigma = min_sigma
        self.relative = relative
        self.epsilon = 1e-3
        self.prediction_type = prediction_type
        self._engine: Optional[Engine] = None
        self._engine_key = None
        self.requires_grad_(False)
        self.eval()

    # ---------------------------------------------------------------------------------------------------------------
    @property
    def device(self):
        return self.transformer.device

    @property
    def dtype(self):
        return self.transformer.dtype

    @property
    def mmdit_precision(self) -> str:
        return self.transformer.mmdit_precision

    @mmdit_precision.setter
    def mmdit_precision(self, value: str) -> None:
        self.transformer.mmdit_precision = value

    def get_engine(self) -> Engine:
        key_t = (self.transformer._weights_key(), self.min_sigma, self.relative, self.prediction_type, self.mmdit_precision)
        key_p = self.time_predictor._weights_key()
        if self._engine is None or key_t != self._engine_key[0]:
            self._engine = Engine(self.transformer.engine_config(), self.device, transformer_sd=self.transformer.state_dict(),
                                  transformer_cfg=self.transformer.config, tpm_sd=self.time_predictor.state_dict(),
                                  min_sigma=self.min_sigma, relative=self.relative, prediction_type=self.prediction_type,
                                  epsilon=self.epsilon, tpm_epsilon=self.time_predictor.epsilon,
                                  tpm_channels=self.time_predictor.conv_out_channels, mmdit_precision=self.mmdit_precision)
        elif key_p != self._engine_key[1]:
            # only the TimePredictor changed (an optimizer step): refresh its packed tensors in place, keep the 4 GB MMDiT pack
            self._engine.refresh_time_predictor(self.time_predictor.state_dict())
        self._engine_key = (key_t, key_p)
        return self._engine

    def encode_prompt(self, prompt=None, negative_prompt=None, num_images_per_prompt: int = 1, device=None, **unused):
        """Reference signature (modeling_sd3_pnt.py:296-380) for the ``pre_process`` hand-over: the three text towers are
        outside this package, so prompts are resolved through ``self.embedding_cache`` (tpdm_b200/embed_cache.py)."""
        cache = getattr(self, "embedding_cache", None)
        if cache is None:
            raise NotImplementedError(
                "text encoders (CLIP-L, CLIP-G, T5-XXL) are outside the tpdm_b200 hot path: pass prompt_embeds, "
                "negative_prompt_embeds, pooled_prompt_embeds and negative_pooled_prompt_embeds, or attach a "
                "PromptEmbeddingCache as model.embedding_cache (SURVEY.md section 8f)")
        if prompt is None:
            raise ValueError("prompt or prompt_embeds must be given")
        prompts = [prompt] if isinstance(prompt, str) else list(prompt)
        negs = negative_prompt if negative_prompt is not None else ""
        negs = [negs] * len(prompts) if isinstance(negs, str) else list(negs)
        if len(negs) != len(prompts):
            raise ValueError(f"negative_prompt has batch size {len(negs)}, prompt has {len(prompts)}")   # :367-372
        device = device or self.device
        pe, pp = cache.get_batch(prompts, device=device)
        ne, np_ = cache.get_batch(negs, device=device)
        rep = lambda t: t.repeat_interleave(num_images_per_prompt, dim=0) if num_images_per_prompt > 1 else t
        return rep(pe), rep(ne), rep(pp), rep(np_)

    def prepare_latents(self, batch_size, num_channels_latents, height, width, dtype, device, generator, latents=None):
        if latents is not None:
            return latents.to(device=device, dtype=dtype)
        shape = (batch_size, num_channels_latents, int(height) // self.vae_scale_factor, int(width) // self.vae_scale_factor)
        # diffusers.utils.torch_utils.randn_tensor semantics: a CPU generator draws on the CPU, then the tensor is moved
        gen = generator[0] if isinstance(generator, (list, tuple)) else generator
        gen_device = gen.device if gen is not None else torch.device(device)
        if gen_device.type != torch.device(device).type:
            return torch.randn(shape, generator=gen, device=gen_device, dtype=dtype).to(device)
        return torch.randn(shape, generator=gen, device=device, dtype=dtype)

    @torch.no_grad()
    def forward(
        self,
        prompt: Union[str, List[str]] = None,
        negative_prompt: Union[str, List[str]] = None,
        prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_prompt_embeds: Optional[torch.FloatTensor] = None,
        pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        num_images_per_prompt: int = 1,
        max_inference_steps: int = 28,
        guidance_scale: Union[float, None] = 7.0,
        generator: Union[torch.Generator, List[torch.Generator]] = None,
        latents: Optional[torch.FloatTensor] = None,
        fix_sigmas: Optional[torch.FloatTensor] = None,
        return_full_process_images: bool = False,
        predict: bool = False,
        ratios: Optional[torch.Tensor] = None,
        return_velocities: bool = False,
        output_type: str = "pil",
        return_hidden_states: Optional[bool] = None,
    ) -> CustomDiffusionModelOutput:
        """Reference signature (modeling_sd3_pnt.py:447-463) + additions: ``output_type`` ("pil" as the reference's
        image_processor.postprocess, "uint8" device tensors (1, H, W, 3), "pt" fp32 (1, 3, H, W)) for the images and:
        ``ratios`` (B, max_inference_steps): Beta draws to inject when predict=False so that two implementations follow
        one trajectory; when omitted the draws are made on the device (the reference calls ``beta_dist.sample()``, :569),
        seeded from ``generator``.  ``return_velocities`` records the per-step CFG velocity (parity tests).
        ``return_hidden_states``: the reference always returns ``hidden_states_combineds`` (:553, 623, one 25 MB D2H copy per
        sample and step); here they stay on the device and are recorded by default only for rollouts (predict=False), which is
        what ``only_predict_logprobs`` replays -- pass True to get them for predict=True as well."""
        if prompt_embeds is None:
            prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds = self.encode_prompt(
                prompt=prompt, negative_prompt=negative_prompt, num_images_per_prompt=num_images_per_prompt)
        if guidance_scale is None:
            raise ValueError("guidance_scale=None is unsupported (as in the reference, whose sigma.repeat(2) is unconditional, :526)")
        if negative_prompt_embeds is None or negative_pooled_prompt_embeds is None or pooled_prompt_embeds is None:
            raise ValueError("negative_prompt_embeds, pooled_prompt_embeds and negative_pooled_prompt_embeds are required")
        device = self.device
        batch_size = prompt_embeds.shape[0]
        side = self.default_sample_size * self.vae_scale_factor
        if latents is None:
            latents = self.prepare_latents(batch_size, self.transformer.config.in_channels, side, side, prompt_embeds.dtype, device,
                                           generator, None)
        init_noise_latents = latents.clone()
        if fix_sigmas is not None:
            max_inference_steps = len(fix_sigmas[0])
        seed = 0
        if not predict and ratios is None:
            # beta_dist.sample() (:569) consumes RNG state: draw the Philox seed of this call FROM the generator, so that a
            # generator reused for several rollouts gives independent schedules (and the same generator state, the same ones)
            gen = generator[0] if isinstance(generator, (list, tuple)) else generator
            seed = int(torch.randint(0, 2**62, (1,), generator=gen, device=gen.device if gen is not None else "cpu").item())
        eng = self.get_engine()
        res = eng.sample(latents, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds,
                         max_inference_steps, float(guidance_scale), bool(predict), ratios=ratios, seed=seed,
                         record_tpm_inputs=(not predict) if return_hidden_states is None else bool(return_hidden_states),
                         record_velocity=return_velocities)
        out_dtype = latents.dtype
        prob_masks = res["prob_masks"]
        logprobs = torch.masked_fill(res["logprobs_raw"], prob_masks, 1.0)          # INVALID_LOGPROB (:615-621)
        hist = res["history_latents"]                                              # (B, T, C, h, w)
        last_valid_indices = []
        finals = []
        for i in range(batch_size):                                                # :646-652
            lv = torch.where(~prob_masks[i])[0][-1]
            last_valid_indices.append(lv)
            finals.append(hist[i, lv])
        finals = torch.stack(finals).to(out_dtype)
        images = []
        if return_full_process_images:                                             # :627-643: every step of every prompt
            if self.vae is None or not hasattr(self.vae, "decode_latents"):
                raise ValueError("return_full_process_images needs the native VAE decoder (pass vae_config or a checkpoint with vae/)")
            for i in range(batch_size):
                steps_i = self.vae.decode_latents(hist[i].to(out_dtype), output_type)   # (T, ...) all recorded steps
                images.append(list(steps_i) if output_type == "pil" else steps_i)
        else:
            images = self._final_images(finals, output_type)
        hcs = None
        if "tpm_inputs_nhwc" in res:  # (B, T, g, g, 2D) bf16 -> reference layout (B, T, 2D, g, g) as a zero-copy view
            hcs = res["tpm_inputs_nhwc"].permute(0, 1, 4, 2, 3)
        out = CustomDiffusionModelOutput(
            init_noise_latents=init_noise_latents, hidden_states_combineds=hcs, tembs=res["tembs"].to(out_dtype), images=images,
            last_valid_indices=last_valid_indices, alphas=res["alphas"], betas=res["betas"], sigmas=res["sigmas"],
            logprobs=logprobs, prob_masks=prob_masks, latents=finals)
        if return_velocities:
            out["velocities"] = res["velocities"]
        return out

    def _final_images(self, finals, output_type):
        """:645-655: the final latent of every prompt through the native decoder (one call) or a caller-supplied module;
        [] without a VAE."""
        images = []
        if self.vae is not None and hasattr(self.vae, "decode_latents"):
            decoded = self.vae.decode_latents(finals, output_type)
            images = [[im] for im in decoded] if output_type == "pil" else [decoded[i:i + 1] for i in range(finals.shape[0])]
        elif self.vae is not None and hasattr(self.vae, "decode"):
            for i in range(finals.shape[0]):
                lat = (finals[i] / self.vae.config.scaling_factor) + self.vae.config.shift_factor
                images.append(self.vae.decode(lat.unsqueeze(0).to(self.vae.dtype), return_dict=False)[0].detach())
        return images

    # ---------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def sample_rollouts(self, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds, latents=None, *,
                        slots: int, max_inference_steps: int = 28, guidance_scale: float = 7.0, generator=None, ratios=None,
                        return_hidden_states: bool = True, output_type: str = "pil", use_graph: bool = True) -> CustomDiffusionModelOutput:
        """Sampled rollouts (``forward(predict=False)``) through the device-side prompt queue: ``slots`` prompts are in flight and
        a prompt leaves its slot when its own trajectory ends, where the lockstep batch of ``forward`` keeps stepping every
        sample until the longest one is done.  ``generator`` is consumed as ``forward`` consumes it (initial latents, then one
        Philox seed), so with equal generator states prompt p gets the rollout ``forward`` gives row p of one batch of all
        prompts: the same Beta draws (or the injected ``ratios`` (P, max_inference_steps)), per-step records and output
        container, with T the longest rollout's step count.  Records past a prompt's last step are zero.  Adds ``steps`` (P,)
        and ``device_steps`` (queue steps executed)."""
        if guidance_scale is None:
            raise ValueError("guidance_scale=None is unsupported (as in the reference, whose sigma.repeat(2) is unconditional, :526)")
        P = prompt_embeds.shape[0]
        side = self.default_sample_size * self.vae_scale_factor
        if latents is None:
            latents = self.prepare_latents(P, self.transformer.config.in_channels, side, side, prompt_embeds.dtype, self.device, generator, None)
        init_noise_latents = latents.clone()
        seed = 0
        if ratios is None:      # the draw forward(predict=False) makes (:292-296)
            gen = generator[0] if isinstance(generator, (list, tuple)) else generator
            seed = int(torch.randint(0, 2**62, (1,), generator=gen, device=gen.device if gen is not None else "cpu").item())
        res = self.get_engine().sample_queue(latents, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds,
                                             int(slots), int(max_inference_steps), float(guidance_scale), use_graph=use_graph, predict=False,
                                             seed=seed, ratios=ratios, record=bool(return_hidden_states))
        steps = res["steps"]
        T = int(steps.max())
        out_dtype = latents.dtype
        prob_masks = torch.arange(T, device=steps.device)[None, :] >= steps[:, None]
        logprobs = torch.masked_fill(res["logprobs_raw"][:, :T], prob_masks, 1.0)          # INVALID_LOGPROB (:615-621)
        finals = res["latents"].to(out_dtype)
        hcs = None
        if "tpm_inputs_nhwc" in res:  # (P, T, g, g, 2D) bf16 -> reference layout (P, T, 2D, g, g) as a zero-copy view
            hcs = res["tpm_inputs_nhwc"][:, :T].permute(0, 1, 4, 2, 3)
        return CustomDiffusionModelOutput(
            init_noise_latents=init_noise_latents, hidden_states_combineds=hcs, tembs=res["tembs"][:, :T].to(out_dtype).contiguous(),
            images=self._final_images(finals, output_type), last_valid_indices=list(steps.long() - 1),
            alphas=res["alphas"][:, :T].contiguous(), betas=res["betas"][:, :T].contiguous(), sigmas=res["sigmas"][:, 1:T + 1].contiguous(),
            logprobs=logprobs, prob_masks=prob_masks, latents=finals, steps=steps, device_steps=res["device_steps"])

    @torch.no_grad()
    def sample_queue(self, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds, latents=None,
                     slots: int = 2, max_inference_steps: int = 28, guidance_scale: float = 7.0, generator=None, ticket=None,
                     decode: bool = False, output_type: str = "pil", use_graph: bool = True, schedule: str = "fifo"):
        """Many prompts with different trajectory lengths on one GPU (BASELINE config 3): ``slots`` prompts are in flight, a
        finished one is replaced on the device from a ticket counter (which several GPUs may share).  Each prompt follows
        exactly the trajectory ``forward(..., predict=True)`` gives it with batch size 1.  Returns a
        CustomDiffusionModelOutput with ``latents`` (P, C, h, w), ``steps`` (P,), ``sigmas`` (P, max_steps + 1) and, with
        ``decode=True`` and a VAE, ``images``."""
        P = prompt_embeds.shape[0]
        side = self.default_sample_size * self.vae_scale_factor
        if latents is None:
            latents = self.prepare_latents(P, self.transformer.config.in_channels, side, side, prompt_embeds.dtype, self.device, generator, None)
        res = self.get_engine().sample_queue(latents, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds,
                                             negative_pooled_prompt_embeds, int(slots), int(max_inference_steps), float(guidance_scale),
                                             ticket=ticket, use_graph=use_graph, schedule=schedule)
        images = []
        if decode and self.vae is not None and hasattr(self.vae, "decode_latents"):
            mine = (res["steps"] > 0).nonzero().flatten().tolist()
            images = {i: self.vae.decode_latents(res["latents"][i: i + 1], output_type) for i in mine}
        return CustomDiffusionModelOutput(
            init_noise_latents=latents, hidden_states_combineds=None, tembs=None, images=images, last_valid_indices=[], alphas=None,
            betas=None, sigmas=res["sigmas"], logprobs=None, prob_masks=None, latents=res["latents"], steps=res["steps"],
            device_steps=res["device_steps"])

    def open_prompt_stream(self, slots: int, capacity: int, max_inference_steps: int = 28, guidance_scale: float = 7.0,
                           use_graph: bool = True, n_text: int = 333):
        """An open prompt queue for serving (engine.PromptStream): ``slots`` prompts in flight, up to ``capacity`` admitted and
        not yet collected.  ``submit`` admits prompts while it runs (latents drawn as ``forward`` draws them when not given),
        ``step`` runs denoising steps, ``results`` returns the finished requests; each gets what ``forward(predict=True)`` with
        batch size 1 gives it.  ``n_text`` is the text length of every prompt (333 for SD3's CLIP + T5 embeddings)."""
        if guidance_scale is None:
            raise ValueError("guidance_scale=None is unsupported (as in the reference, whose sigma.repeat(2) is unconditional, :526)")
        side = self.default_sample_size * self.vae_scale_factor
        C = self.transformer.config.in_channels
        draw = lambda n, generator, dtype: self.prepare_latents(n, C, side, side, dtype, self.device, generator, None)
        return self.get_engine().open_stream(int(slots), int(capacity), int(max_inference_steps), float(guidance_scale), use_graph,
                                             latent=side // self.vae_scale_factor, n_text=int(n_text), prepare_latents=draw)

    # ---------------------------------------------------------------------------------------------------------------
    def _replay_trainer(self, grid: int, samples: int):
        """TimePredictorTrainer (native forward with saved activations + backward) behind the differentiable replay."""
        from .tpm_training import TimePredictorTrainer

        tr = getattr(self, "_replay", None)
        if tr is None or tr.g != grid or tr.max_samples < samples or tr.module is not self.time_predictor:
            self._replay = None          # release the old workspace first
            tr = self._replay = TimePredictorTrainer(self.time_predictor, grid, samples)
        return tr

    def only_predict_logprobs(self, fix_sigmas: torch.Tensor, fix_hidden_states_combineds: torch.Tensor, fix_tembs: torch.Tensor):
        """modeling_sd3_pnt.py:670-726.  With autograd enabled and a trainable ``time_predictor`` (the RLOO wrapper, :760-763) the
        result carries a grad_fn whose backward is the native TimePredictor backward and deposits ``time_predictor.*.grad``, so
        ``loss.backward()`` in the reference trainer (rloo_trainer.py:485-501) works on the drop-in; otherwise a plain replay."""
        from . import _lib as L

        if fix_sigmas is None:
            raise ValueError("fix_sigmas must be provided")
        if fix_hidden_states_combineds is None:
            raise ValueError("fix_hidden_states_combineds must be provided")
        device = self.device
        batch_size, steps = fix_sigmas.shape[:2]
        ptype = self.prediction_type
        hcs = fix_hidden_states_combineds.to(device)                 # the reference keeps them on the CPU (:553, :689)
        tembs = fix_tembs.to(device)
        g = hcs.shape[-1]
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.time_predictor.parameters()):
            x_nhwc = hcs.permute(0, 1, 3, 4, 2)                      # a view of the NHWC storage forward() recorded
            tr = self._replay_trainer(g, batch_size * steps)
            lp = tr.logprobs(fix_sigmas, x_nhwc, tembs, self.min_sigma, self.epsilon, self.relative, ptype)
            return {"logprobs": lp}
        with torch.no_grad():
            eng = self.get_engine()
            ab = torch.stack([eng.tpm_forward(hcs[:, step], tembs[:, step]) for step in range(steps)], dim=1).contiguous()   # (B, T, 2)
            sig = fix_sigmas.to(device=device, dtype=torch.float32).contiguous()
            lp = torch.empty(batch_size, steps, device=device, dtype=torch.float32)
            with torch.cuda.device(device):
                L.check(L.load().tpdm_beta_logprob(L.ptr(ab), L.ptr(sig), batch_size, steps, float(self.min_sigma), float(self.epsilon),
                                                   1 if self.relative else 0, 0 if ptype == "alpha_beta" else 1,
                                                   float(self.time_predictor.epsilon), L.ptr(lp), None, L.stream_ptr()))
        return {"logprobs": lp}


class SD3PredictNextTimeStepModelRLOOWrapper(nn.Module):
    """modeling_sd3_pnt.py:729-933: the surface CommonRLOOTrainer calls (rloo_trainer.py:432-485)."""

    def __init__(
        self,
        pretrained_model_name_or_path=None,
        torch_dtype: torch.dtype = torch.float16,
        min_sigma: float = 0.01,
        pre_process: bool = False,
        init_alpha: float = 1.5,
        init_beta: float = 0.5,
        relative: bool = True,
        prediction_type: str = "alpha_beta",
        fsdp: str = [],
        max_inference_steps: int = 28,
        transformer_config: Optional[dict] = None,
        device=None,
        mmdit_precision: str = "bf16",
    ):
        super().__init__()
        self.pretrained_model_name_or_path = pretrained_model_name_or_path or ""
        self.agent_model = SD3PredictNextTimeStepModel(
            pretrained_model_name_or_path, torch_dtype=torch_dtype, init_alpha=init_alpha, init_beta=init_beta, min_sigma=min_sigma,
            pre_process=pre_process, relative=relative, prediction_type=prediction_type, transformer_config=transformer_config,
            device=device, mmdit_precision=mmdit_precision).eval()
        self.relative = relative
        self.fsdp = fsdp
        self.max_inference_steps = max_inference_steps
        self.agent_model.requires_grad_(False)
        self.agent_model.time_predictor.train()
        self.agent_model.time_predictor.requires_grad_(True)

    def rloo_repeat(self, data, rloo_k):
        """:768-786"""
        if "prompt" in data:
            data["prompt"] = data["prompt"] * rloo_k
        for key in ["prompt_embeds", "negative_prompt_embeds", "pooled_prompt_embeds", "negative_pooled_prompt_embeds"]:
            if key in data:
                size = [rloo_k] + [1] * (len(data[key].shape) - 1)
                data[key] = data[key].repeat(*size)
        return data

    def sample(self, inputs):
        """:788-806 (weights are replicated per GPU, so there is no FSDP summon)."""
        if "3.5" in self.pretrained_model_name_or_path:
            inputs["guidance_scale"] = 3.5
        inputs["max_inference_steps"] = self.max_inference_steps
        return self.agent_model(**{k: v for k, v in inputs.items() if k != "prompt" or "prompt_embeds" not in inputs})

    def reward(self, inputs, outputs, reward_model, gamma=0.8, return_last_reward=False):
        """:808-849.  ``reward_model.score(prompt, image)`` is caller-supplied (reward towers are out of scope); when the
        pipeline has no VAE the final latent (C, h, w) is handed to it in place of the PIL image."""
        prompts = inputs.get("prompt", None)
        images = outputs.get("images", None)
        prob_masks = outputs.get("prob_masks", None)
        last_valid_indices = outputs.get("last_valid_indices", [])
        if not images:
            images = [[lat] for lat in outputs["latents"]]
        if prompts is None or images is None:
            raise ValueError("prompt and images must be provided")
        elif len(prompts) != len(images):
            raise ValueError("prompt and images must have the same length")
        rewards, last_image_rewards = [], []
        for i, (prompt, image, prob_mask) in enumerate(zip(prompts, images, prob_masks)):
            if last_valid_indices == []:
                last_image_idx = torch.where(~prob_mask.bool())[-1][-1].item()
                last_image = image[last_image_idx]
            else:
                last_image_idx = int(last_valid_indices[i])
                last_image = image[0]
            last_image_reward = float(reward_model.score(prompt, last_image))
            last_image_rewards.append(last_image_reward)
            reward = 0
            for j in range(last_image_idx + 1):
                reward += last_image_reward * (gamma ** (last_image_idx - j))
            rewards.append(reward / (last_image_idx + 1))
        rewards, last_image_rewards = torch.tensor(rewards), torch.tensor(last_image_rewards)
        return (rewards, last_image_rewards) if return_last_reward else rewards

    def logprobs(self, inputs, outputs):
        """:851-873"""
        return self.agent_model.only_predict_logprobs(
            fix_sigmas=outputs["sigmas"], fix_hidden_states_combineds=outputs["hidden_states_combineds"],
            fix_tembs=outputs["tembs"])["logprobs"]

    def kl_divergence(self, outputs: CustomDiffusionModelOutput):
        """:875-901 on the device: KL(Beta(alpha, beta) || reference Beta) per step, 0 where masked -> (bs, T)."""
        from .rloo import shape_rollout
        return shape_rollout(outputs, None, relative=self.relative)["kl"]

    def subset_inputs(self, inputs, micro_batch_inds):
        """:903-914"""
        subset = {}
        for key, value in inputs.items():
            if isinstance(value, torch.Tensor):
                subset[key] = value[micro_batch_inds]
            elif isinstance(value, list):
                subset[key] = [value[i] for i in micro_batch_inds]
            elif isinstance(value, (float, int)) or value is None:
                subset[key] = value
            else:
                raise ValueError(f"Unsupported input type: {type(value)}")
        return subset

    def subset_outputs(self, outputs, micro_batch_inds):
        """:916-933"""
        subset = {}
        for key, value in outputs.items():
            if isinstance(value, torch.Tensor):
                subset[key] = value[micro_batch_inds]
            elif isinstance(value, list):
                subset[key] = [value[i] for i in micro_batch_inds] if len(value) else []    # `images` is empty without a VAE
            elif isinstance(value, dict):
                subset[key] = {k: v[micro_batch_inds] for k, v in value.items() if isinstance(v, torch.Tensor)}
            elif value is None:
                subset[key] = None
            else:
                raise ValueError(f"Unsupported output type: {type(value)}")
        return subset
