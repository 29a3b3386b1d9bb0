"""bf16 against the opt-in FP8 mode (mmdit_precision="fp8": QKV and FF1 as E4M3 GEMMs) on the SD3-medium 1024^2 trajectory,
B = 1, in one process with the same weights.  The two models alternate for several rounds of back-to-back trajectories (at
least `seconds` per variant and round) under the power cap, as tools/sustained_steps.py runs them; reported are the median
and spread of ms per denoising step and images/s, the median SM clock and power while each variant ran, the GEMM-class device
time of one trajectory (tpdm_profile_*), and stand-alone TFLOP/s of the QKV and FF1 GEMM shapes of a step in both precisions.
The card name, power limit and maximum SM clock are read in the same run.

    python tools/fp8_steps.py [--seconds 8] [--rounds 4] [--out profiles/fp8_steps_n1.json]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tpdm_b200 import _lib as L  # noqa: E402
from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel  # noqa: E402


def smi(query):
    r = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True)
    return [s.strip() for s in r.stdout.strip().split(",")]


class Sampler:
    """SM clock and power draw every 0.25 s while a variant runs."""

    def __init__(self):
        self.samples, self.stop = [], False
        self.th = threading.Thread(target=self.run, daemon=True)
        self.th.start()

    def run(self):
        while not self.stop:
            try:
                c, p = smi("clocks.sm,power.draw")
                self.samples.append((float(c), float(p)))
            except Exception:
                pass
            time.sleep(0.25)

    def finish(self):
        self.stop = True
        self.th.join()
        med = lambda i: statistics.median(s[i] for s in self.samples) if self.samples else float("nan")
        return med(0), med(1)


def sustained(model, kw, seconds):
    for _ in range(2):
        model(**kw, max_inference_steps=28, predict=True)
    torch.cuda.synchronize()
    smp = Sampler()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    steps, images, t0 = 0, 0, time.perf_counter()
    e0.record()
    while time.perf_counter() - t0 < seconds:
        out = model(**kw, max_inference_steps=28, predict=True)
        steps += int(out.sigmas.shape[1])
        images += 1
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clk, pw = smp.finish()
    return dict(ms_per_step=ms / steps, images_per_s=images / ms * 1e3, steps=steps, images=images, sm_clock_mhz=clk, power_w=pw)


def gemm_class_time(model, kw):
    lib = L.load()
    model(**kw, max_inference_steps=28, predict=True)
    torch.cuda.synchronize()
    L.check(lib.tpdm_profile_start(16384))
    out = model(**kw, max_inference_steps=28, predict=True)
    torch.cuda.synchronize()
    ms, fl, ct = (C.c_double * 4)(), (C.c_double * 4)(), (C.c_longlong * 4)()
    L.check(lib.tpdm_profile_stop(ms, fl, ct, 4))
    steps = int(out.sigmas.shape[1])
    return dict(steps=steps, gemm_ms_per_step=ms[0] / steps, gemm_launches=int(ct[0]), gemm_tflops=fl[0] / (ms[0] * 1e-3) / 1e12,
                class_ms_per_step=dict(gemm=ms[0] / steps, attention=ms[1] / steps, ln_modulate=ms[2] / steps, adaln_gemv=ms[3] / steps))


def gemm_rates(reps=200):
    """Stand-alone rates of the step's QKV (image rows of both CFG halves, plus the text tail) and FF1 + GELU GEMMs."""
    from tpdm_b200.engine import quantize_fp8_rows

    lib = L.load()
    res = {}
    torch.manual_seed(0)
    for name, batch, rows, N, K, epi in (("qkv", 2, 4096, 4608, 1536, 0), ("qkv_text", 2, 333, 4608, 1536, 0), ("ff1_gelu", 2, 4096, 6144, 1536, 2)):
        A = torch.randn(batch, rows, K, device="cuda")
        W = torch.randn(N, K, device="cuda") * 0.03
        bias = torch.zeros(N, device="cuda")
        out = torch.empty(batch, rows, N, device="cuda", dtype=torch.bfloat16)
        a16, w16 = A.bfloat16(), W.bfloat16()
        a8, a_s = quantize_fp8_rows(A.reshape(-1, K))
        w8, w_s = quantize_fp8_rows(W)
        runs = {
            "bf16": lambda: lib.tpdm_gemm_bf16(L.ptr(a16), L.ptr(w16), L.ptr(bias), None, L.ptr(out), batch, rows, N, K, epi, None),
            "fp8": lambda: lib.tpdm_gemm_fp8(L.ptr(a8), L.ptr(a_s), L.ptr(w8), L.ptr(w_s), L.ptr(bias), L.ptr(out), batch, rows, N, K, epi, None),
        }
        flops = 2.0 * batch * rows * N * K
        for prec, fn in runs.items():
            for _ in range(10):
                L.check(fn())
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / reps
            res[f"{name}_{prec}"] = dict(shape=[batch, rows, N, K], us=us, tflops=flops / (us * 1e-6) / 1e12)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--out", default="profiles/fp8_steps_n1.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fp8_steps.py measures on the GPU; no CUDA device found")
    name, plimit, maxclk = smi("name,power.limit,clocks.max.sm")
    torch.manual_seed(1234)
    models = {}
    for prec in ("bf16", "fp8"):
        m = SD3PredictNextTimeStepModel(transformer_config=SD3_MEDIUM_TRANSFORMER_CONFIG, torch_dtype=torch.bfloat16, device="cuda",
                                        mmdit_precision=prec)
        if models:
            m.load_state_dict(models["bf16"].state_dict())
        models[prec] = m
    g = torch.Generator().manual_seed(0)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    kw = dict(prompt_embeds=mk(1, 333, 4096), negative_prompt_embeds=mk(1, 333, 4096), pooled_prompt_embeds=mk(1, 2048),
              negative_pooled_prompt_embeds=mk(1, 2048), latents=mk(1, 16, 128, 128))
    rates = gemm_rates()
    prof = {p: gemm_class_time(m, kw) for p, m in models.items()}
    rounds = {p: [] for p in models}
    for r in range(a.rounds):
        order = ("bf16", "fp8") if r % 2 == 0 else ("fp8", "bf16")
        for p in order:
            rounds[p].append(sustained(models[p], kw, a.seconds))
            print(f"round {r} {p}: {rounds[p][-1]}", flush=True)
    summary = {}
    for p, rs in rounds.items():
        ms = [x["ms_per_step"] for x in rs]
        ips = [x["images_per_s"] for x in rs]
        summary[p] = dict(ms_per_step_median=statistics.median(ms), ms_per_step_min=min(ms), ms_per_step_max=max(ms),
                          images_per_s_median=statistics.median(ips), sm_clock_mhz_median=statistics.median(x["sm_clock_mhz"] for x in rs),
                          power_w_median=statistics.median(x["power_w"] for x in rs))
    summary["step_time_change"] = summary["fp8"]["ms_per_step_median"] / summary["bf16"]["ms_per_step_median"] - 1.0
    res = dict(card=name, power_limit_w=float(plimit), max_sm_clock_mhz=float(maxclk), workload="SD3-medium 1024^2, B=1, CFG 7, predict=True, "
               "reference TimePredictor init, 28-step cap", seconds_per_variant_and_round=a.seconds, rounds=rounds, summary=summary,
               gemm_profile=prof, standalone_gemm=rates)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(summary=summary, standalone={k: round(v["tflops"]) for k, v in rates.items()},
                          gemm_ms_per_step={p: v["gemm_ms_per_step"] for p, v in prof.items()}, card=name, power_limit_w=plimit), indent=1))


if __name__ == "__main__":
    main()
