"""Minimal RLOO update around the native pieces: the arithmetic of CommonRLOOTrainer.train for ONE update
(/root/reference/src/train/rloo_trainer.py:425-523) without the HF Trainer / trl / accelerate plumbing (out of scope,
SURVEY.md section 2.1 #6).  rollout (device-side Beta draws) -> reward -> RLOO advantage -> PPO epochs over micro-batches ->
native TPM backward + flat-buffer all-reduce + fused AdamW."""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import torch

from .tpm_training import TimePredictorTrainer


def shape_rollout(outputs: Dict, last_rewards: Optional[torch.Tensor] = None, *, relative: bool = True, gamma: float = 0.97,
                  kl_coef: float = 0.0, mean_kl: bool = False, rloo_k: int = 0, ref_steps: int = 28) -> Dict[str, torch.Tensor]:
    """Device-side reward shaping of one rollout (C ABI ``tpdm_rollout_shaping``): per-step KL to the reference schedule
    (modeling_sd3_pnt.py:875-901), discounted score (:828-841), ``rlhf_reward = score - kl_coef * kl`` and the RLOO
    leave-one-out advantage (rloo_trainer.py:447-461).  ``last_rewards`` (B,) is the caller's reward-model score of each
    final image; ``rloo_k = 0`` skips the advantage."""
    from . import _lib as L
    lib = L.load()
    alphas = outputs["alphas"].float().contiguous()
    if not alphas.is_cuda:
        raise RuntimeError("shape_rollout needs the rollout tensors on the CUDA device (there is no CPU path)")
    dev = alphas.device
    betas, sigmas = outputs["betas"].float().contiguous(), outputs["sigmas"].float().contiguous()
    masks = outputs["prob_masks"].to(device=dev, dtype=torch.int32).contiguous()
    B, T = alphas.shape
    lr = None if last_rewards is None else last_rewards.to(device=dev, dtype=torch.float32).contiguous()
    kl = torch.empty(B, T, device=dev)
    scores, rlhf = torch.empty(B, device=dev), torch.empty(B, device=dev)
    adv = torch.empty(B, device=dev) if rloo_k else None
    with torch.cuda.device(dev):
        L.check(lib.tpdm_rollout_shaping(L.ptr(alphas), L.ptr(betas), L.ptr(sigmas), L.ptr(masks), L.ptr(lr) if lr is not None else None,
                                         B, T, 1 if relative else 0, ref_steps, gamma, kl_coef, 1 if mean_kl else 0, int(rloo_k),
                                         L.ptr(kl), L.ptr(scores), L.ptr(rlhf), L.ptr(adv) if adv is not None else None,
                                         torch.cuda.current_stream().cuda_stream))
    return dict(kl=kl, scores=scores, rlhf_reward=rlhf, advantages=adv)


def rloo_advantages(rlhf_reward: torch.Tensor, rloo_k: int) -> torch.Tensor:
    """rloo_trainer.py:458-461 (layout = rloo_k repeats x prompts, as rloo_repeat tiles the prompt list)."""
    r = rlhf_reward.reshape(rloo_k, -1)
    baseline = (r.sum(0) - r) / (rloo_k - 1)
    return (r - baseline).flatten()


def rloo_update(wrapper, trainer: TimePredictorTrainer, data: Dict, reward_fn: Callable, rloo_k: int = 2, num_ppo_epochs: int = 4,
                micro_batch_size: int = 8, cliprange: float = 0.2, gamma: float = 0.97, kl_coef: float = 0.0, seed: int = 0,
                generator: Optional[torch.Generator] = None, slots: Optional[int] = None) -> Dict:
    """`wrapper`: SD3PredictNextTimeStepModelRLOOWrapper; `data`: dict with the four embedding tensors (and optionally
    'prompt'); `reward_fn(latents (B,C,h,w), outputs) -> (B,)` stands in for the reward model.  Randomness (initial noise, Beta
    draws, micro-batch permutations) comes from ``generator``, or from one generator per trainer that is seeded with ``seed`` on
    the FIRST update and then keeps advancing, so successive updates see independent rollouts (the reference's global RNG does
    the same, rloo_trainer.py:133).  ``slots=None`` samples the rollouts as one lockstep batch (``wrapper.sample``, the
    reference's semantics: finished samples keep stepping until the longest is done); an integer samples the same rollouts
    through the device-side prompt queue with that many in flight (``sample_rollouts``), where each leaves its slot when it ends."""
    agent = wrapper.agent_model
    data = wrapper.rloo_repeat(dict(data), rloo_k)
    if generator is None:
        generator = getattr(trainer, "_rollout_generator", None)
        if generator is None:
            generator = trainer._rollout_generator = torch.Generator().manual_seed(seed)
    if slots is None:
        outputs = wrapper.sample({**data, "predict": False, "generator": generator})
    else:
        guidance = 3.5 if "3.5" in wrapper.pretrained_model_name_or_path else data.get("guidance_scale", 7.0)     # as wrapper.sample
        outputs = agent.sample_rollouts(data["prompt_embeds"], data["negative_prompt_embeds"], data["pooled_prompt_embeds"],
                                        data["negative_pooled_prompt_embeds"], data.get("latents"), slots=slots,
                                        max_inference_steps=wrapper.max_inference_steps, guidance_scale=guidance, generator=generator)
    prob_masks = outputs["prob_masks"]
    last_reward = reward_fn(outputs["latents"], outputs).float()
    shaped = shape_rollout(outputs, last_reward, relative=agent.relative, gamma=gamma, kl_coef=kl_coef, rloo_k=rloo_k)
    scores, advantages = shaped["scores"].cpu(), shaped["advantages"]
    B = scores.shape[0]
    x = outputs["hidden_states_combineds"].permute(0, 1, 3, 4, 2)     # back to the NHWC storage it is a view of
    logs: List[Dict] = []
    for _ in range(num_ppo_epochs):
        perm = torch.randperm(B, generator=generator).numpy()
        for s in range(0, B, micro_batch_size):
            idx = torch.as_tensor(perm[s: s + micro_batch_size], device=agent.device)
            st = trainer.ppo_update(outputs["sigmas"][idx], outputs["logprobs"][idx], x[idx], outputs["tembs"][idx], advantages[idx],
                                    min_sigma=agent.min_sigma, cliprange=cliprange, epsilon=agent.epsilon, relative=agent.relative,
                                    prediction_type=agent.prediction_type)
            logs.append({k: float(v) for k, v in st.items() if k != "new_logprobs"})
    trainer.sync_to_module()
    return dict(scores=scores, advantages=advantages.cpu(), steps=(~prob_masks).sum(1).float().mean().item(), logs=logs)
