"""BASELINE config 4 rollout sampling through the lockstep batch and through the device-side prompt queue, on one GPU.

SD3-medium at 512^2, 4 seeded prompts x rloo_k 4 = 16 rollouts, init_alpha 2.5, init_beta 1.0, min_sigma 0.01, at most 28 steps
(launch_sd3_train.sh:16-19, as bench.py --workload config4).  In one process and alternating, every repetition samples the same
rollouts (same generator state) three ways: the lockstep batch ``forward(predict=False)``, which steps every rollout until the
longest is done, and ``sample_rollouts`` with 16 and with 8 queue slots, where a rollout leaves its slot when it ends.  Then whole
``rloo_update`` calls with and without ``slots`` alternate.  Times are CUDA events around each call.  Prints one JSON object and
writes it to ``--out`` when given.

    python tools/rollout_queue.py [--reps 5] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModelRLOOWrapper  # noqa: E402
from tpdm_b200.rloo import rloo_update  # noqa: E402
from tpdm_b200.tpm_training import TimePredictorTrainer  # noqa: E402

PROMPTS, RLOO_K, MAX_STEPS, N_TEXT = 4, 4, 28, 333


def gpu_info(dev: torch.device) -> dict:
    r = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, limit, clock = (r.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return dict(name=name or torch.cuda.get_device_name(dev), power_limit=limit, max_sm_clock=clock)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)
    cfg = dict(SD3_MEDIUM_TRANSFORMER_CONFIG, sample_size=64)
    wrapper = SD3PredictNextTimeStepModelRLOOWrapper(transformer_config=cfg, torch_dtype=torch.bfloat16, device=dev, min_sigma=0.01,
                                                     init_alpha=2.5, init_beta=1.0, max_inference_steps=MAX_STEPS)
    agent = wrapper.agent_model
    g = torch.Generator().manual_seed(77)
    mk = lambda *s: torch.randn(*s, generator=g).to(dev)
    data = dict(prompt_embeds=mk(PROMPTS, N_TEXT, 4096), negative_prompt_embeds=mk(PROMPTS, N_TEXT, 4096), pooled_prompt_embeds=mk(PROMPTS, 2048),
                negative_pooled_prompt_embeds=mk(PROMPTS, 2048))
    rep = wrapper.rloo_repeat(dict(data), RLOO_K)
    emb = (rep["prompt_embeds"], rep["negative_prompt_embeds"], rep["pooled_prompt_embeds"], rep["negative_pooled_prompt_embeds"])
    n = PROMPTS * RLOO_K

    modes = {
        "lockstep": lambda gen: wrapper.sample({**rep, "predict": False, "generator": gen}),
        "queue_16_slots": lambda gen: agent.sample_rollouts(*emb, slots=16, max_inference_steps=MAX_STEPS, generator=gen),
        "queue_8_slots": lambda gen: agent.sample_rollouts(*emb, slots=8, max_inference_steps=MAX_STEPS, generator=gen),
    }
    rows = {k: [] for k in modes}
    same_rollouts = True
    for r in range(args.warmup + args.reps):
        steps_of = {}
        for name, fn in modes.items():
            ms, out = timed(lambda: fn(torch.Generator().manual_seed(1000 + r)))
            steps = (~out["prob_masks"]).sum(1)
            T = out["prob_masks"].shape[1]
            steps_of[name] = steps.tolist()
            dsteps = T if name == "lockstep" else int(out["device_steps"])
            if r >= args.warmup:
                rows[name].append(dict(ms=ms, sum_steps=int(steps.sum()), longest=T, lockstep_slot_steps=n * T, device_steps=dsteps))
            del out
        same_rollouts = same_rollouts and len({tuple(v) for v in steps_of.values()}) == 1

    trainer = TimePredictorTrainer(agent.time_predictor, grid=32, max_samples=8 * MAX_STEPS, lr=1e-6, betas=(0.9, 0.99), eps=1e-5)
    reward = lambda latents, outputs: -(latents.float() ** 2).mean(dim=(1, 2, 3))
    upd = {"lockstep": None, "queue_16_slots": 16}
    upd_ms = {k: [] for k in upd}
    for r in range(args.warmup + args.reps):
        for name, slots in upd.items():
            ms, _ = timed(lambda: rloo_update(wrapper, trainer, data, reward, rloo_k=RLOO_K, num_ppo_epochs=4, micro_batch_size=8, cliprange=0.2,
                                              gamma=0.97, generator=torch.Generator().manual_seed(5000 + r), slots=slots))
            if r >= args.warmup:
                upd_ms[name].append(ms)

    med = lambda xs: statistics.median(xs)
    summary = {}
    for name, rs in rows.items():
        summary[name] = dict(ms_per_batch_median=med([x["ms"] for x in rs]), ms_per_batch=[round(x["ms"], 1) for x in rs],
                             sum_steps=[x["sum_steps"] for x in rs], longest=[x["longest"] for x in rs],
                             lockstep_slot_steps=[x["lockstep_slot_steps"] for x in rs], device_steps=[x["device_steps"] for x in rs])
    result = dict(
        workload=f"SD3-medium 512^2 (random init, bf16), {PROMPTS} prompts x rloo_k {RLOO_K} = {n} rollouts, init_alpha 2.5, init_beta 1.0, "
                 f"min_sigma 0.01, <= {MAX_STEPS} steps, device-side Beta draws, seeded embeddings",
        gpu=gpu_info(dev), reps=args.reps, warmup=args.warmup, same_step_counts_in_every_mode=same_rollouts, rollout_sampling=summary,
        rloo_update={k: dict(ms_median=med(v), ms=[round(x, 1) for x in v]) for k, v in upd_ms.items()},
    )
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
