"""The open prompt stream against the closed device-side queue, and as a server on an arrival trace, on one GPU.

SD3-medium 1024^2 (random init, bf16), built and seeded as ``bench.py --workload config3`` builds it: the same model seed,
TimePredictor scaling and per-prompt inputs, so that trajectory lengths vary (the per-prompt step counts and their histogram are
recorded); 32 prompts, 2 slots, at most 28 steps.

(a) against (b), alternating for ``--rounds`` rounds after one warm-up round each: (a) is the closed ``sample_queue`` over all 32
prompts, (b) a stream (capacity 32) with all 32 submitted at open and drained.  Times are CUDA events around each call.  Device
steps are the steps the GPU executed; the closed queue enqueues one more, which the device skips, so (a) counts
``device_steps - 1``.

``--mixed-options`` adds (m), alternating with (a) and (b): the stream of (b) with per-request options -- prompt i gets guidance
(3.5, 5, 7, 9)[i % 4]; prompts with i % 4 == 1 are sampled (predict=False, seed 1000 + i) and those with i % 4 == 2 are capped at
12 steps.  The work per device step is that of (b); only the number of steps differs.

(c) Arrival trace: prompt i arrives at i x ``--interval-factor`` x (a)'s median time per image.  The stream server submits each
prompt when it arrives and steps while anything is in flight; the FIFO server runs batch-1 ``forward(predict=True)`` per request
in arrival order.  Latency is host time from arrival (= submit) to the result being on the host.

Prints one JSON object and writes it to ``--out`` when given.

    python tools/prompt_stream.py [--rounds 4] [--mixed-options] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel  # noqa: E402

PROMPTS, SLOTS, MAX_STEPS, N_TEXT = 32, 2, 28, 333


def gpu_info(dev: torch.device) -> dict:
    r = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, limit, clock, max_clock = (r.stdout.strip().split(", ") + ["?"] * 4)[:4]
    return dict(name=name or torch.cuda.get_device_name(dev), power_limit=limit, sm_clock=clock, max_sm_clock=max_clock)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--interval-factor", type=float, default=1.2)
    ap.add_argument("--mixed-options", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)     # as bench.py build_model: the same random-init weights
    model = SD3PredictNextTimeStepModel(transformer_config=dict(SD3_MEDIUM_TRANSFORMER_CONFIG), torch_dtype=torch.bfloat16, device=dev,
                                        init_alpha=1.5, init_beta=0.5)
    with torch.no_grad():       # as bench.py --workload config3: (alpha, beta) depend on the hidden states
        tp = model.time_predictor
        tp.fc2.weight.mul_(4.0)
        tp.fc1.weight.mul_(4.0)
        tp.conv2.weight.mul_(2.0)

    def prompt(i):              # bench.py run_config3 inputs(i)
        g = torch.Generator().manual_seed(5000 + i)
        mk = lambda *s: torch.randn(*s, generator=g).to(dev)
        return [mk(1, N_TEXT, 4096), mk(1, N_TEXT, 4096), mk(1, 2048), mk(1, 2048), mk(1, 16, 128, 128)]

    cols = list(zip(*[prompt(i) for i in range(PROMPTS)]))
    inp = dict(zip(("prompt_embeds", "negative_prompt_embeds", "pooled_prompt_embeds", "negative_pooled_prompt_embeds", "latents"),
                   [torch.cat(c) for c in cols]))
    emb = (inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["pooled_prompt_embeds"], inp["negative_pooled_prompt_embeds"])

    def closed():
        q = model.sample_queue(*emb, latents=inp["latents"], slots=SLOTS, max_inference_steps=MAX_STEPS)
        return dict(executed=int(q.device_steps) - 1, steps=q.steps.tolist(), latents=q.latents)

    def stream():
        with model.open_prompt_stream(slots=SLOTS, capacity=PROMPTS, max_inference_steps=MAX_STEPS) as s:
            rids = s.submit(*emb, latents=inp["latents"])
            res = s.drain()
            executed = s.device_steps
        return dict(executed=executed, steps=[res[r]["steps"] for r in rids], latents=torch.stack([res[r]["latents"] for r in rids]))

    mixed_opts = dict(guidance_scale=[(3.5, 5.0, 7.0, 9.0)[i % 4] for i in range(PROMPTS)], predict=[i % 4 != 1 for i in range(PROMPTS)],
                      seed=[1000 + i for i in range(PROMPTS)], max_inference_steps=[12 if i % 4 == 2 else MAX_STEPS for i in range(PROMPTS)])

    def stream_mixed():
        with model.open_prompt_stream(slots=SLOTS, capacity=PROMPTS, max_inference_steps=MAX_STEPS) as s:
            rids = s.submit(*emb, latents=inp["latents"], **mixed_opts)
            res = s.drain()
            executed = s.device_steps
        return dict(executed=executed, steps=[res[r]["steps"] for r in rids])

    runs = [("a_closed_queue", closed), ("b_stream", stream)] + ([("m_stream_mixed_options", stream_mixed)] if args.mixed_options else [])
    rows = {name: [] for name, _ in runs}
    agree = []
    for r in range(1 + args.rounds):
        outs = {}
        for name, fn in runs:
            ms, out = timed(fn)
            outs[name] = out
            if r >= 1:
                rows[name].append(dict(ms=ms, executed=out["executed"], ms_per_step=ms / out["executed"], images_per_s=PROMPTS / ms * 1e3))
        a, b = outs["a_closed_queue"], outs["b_stream"]
        agree.append(dict(steps_equal=a["steps"] == b["steps"],
                          latent_rel_l2=float((a["latents"] - b["latents"]).norm() / a["latents"].norm())))
    med = lambda xs: statistics.median(xs)
    ab = {k: dict(device_steps=[x["executed"] for x in v], ms=[round(x["ms"], 1) for x in v], ms_per_step=[round(x["ms_per_step"], 3) for x in v],
                  ms_per_step_median=med([x["ms_per_step"] for x in v]), images_per_s_median=med([x["images_per_s"] for x in v]))
          for k, v in rows.items()}
    ab["b_over_a_ms_per_step"] = ab["b_stream"]["ms_per_step_median"] / ab["a_closed_queue"]["ms_per_step_median"]
    if args.mixed_options:
        ab["m_over_b_ms_per_step"] = ab["m_stream_mixed_options"]["ms_per_step_median"] / ab["b_stream"]["ms_per_step_median"]
        ab["m_steps_per_prompt"] = outs["m_stream_mixed_options"]["steps"]
    ab["agreement"] = agree
    steps = outs["a_closed_queue"]["steps"]
    ab["steps_per_prompt"] = steps
    ab["steps_histogram"] = {str(k): steps.count(k) for k in sorted(set(steps))}
    ab["sum_of_steps"] = sum(steps)

    # (c) arrival trace
    per_image_s = med([x["ms"] for x in rows["a_closed_queue"]]) / PROMPTS / 1e3
    interval = args.interval_factor * per_image_s
    arrivals = [i * interval for i in range(PROMPTS)]
    one = lambda i: {k: v[i:i + 1] for k, v in inp.items()}

    def serve_stream():
        lat = {}
        with model.open_prompt_stream(slots=SLOTS, capacity=PROMPTS, max_inference_steps=MAX_STEPS) as s:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nxt, arrived = 0, {}
            while len(lat) < PROMPTS:
                now = time.perf_counter() - t0
                while nxt < PROMPTS and arrivals[nxt] <= now:
                    (rid,) = s.submit(**one(nxt))
                    arrived[rid] = arrivals[nxt]
                    nxt += 1
                s.step()
                for rid in s.results():
                    lat[rid] = time.perf_counter() - t0 - arrived[rid]
                if len(lat) == len(arrived) and nxt < PROMPTS:      # idle: wait for the next arrival
                    time.sleep(max(0.0, arrivals[nxt] - (time.perf_counter() - t0)))
        return list(lat.values())

    def serve_fifo():
        lat = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(PROMPTS):
            wait = arrivals[i] - (time.perf_counter() - t0)
            if wait > 0:
                time.sleep(wait)
            o = model(**one(i), max_inference_steps=MAX_STEPS, predict=True)
            o.latents.cpu()
            lat.append(time.perf_counter() - t0 - arrivals[i])
        return lat

    serve_fifo()                 # warm the batch-1 plan and its step graphs
    trace = {}
    for name, fn in (("stream", serve_stream), ("fifo_forward", serve_fifo)):
        xs = fn()
        trace[name] = dict(p50_s=pct(xs, 0.5), p90_s=pct(xs, 0.9), max_s=max(xs), mean_s=sum(xs) / len(xs))
    result = dict(
        workload=f"SD3-medium 1024^2 (random init, bf16), bench.py config3 model seed, TimePredictor scaling and inputs, {PROMPTS} prompts, {SLOTS} slots, "
                 f"<= {MAX_STEPS} steps, predict mode",
        gpu=gpu_info(dev), rounds=args.rounds, closed_vs_stream=ab,
        arrival_trace=dict(interval_s=interval, interval_factor=args.interval_factor, per_image_s_closed_queue=per_image_s, **trace),
    )
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
