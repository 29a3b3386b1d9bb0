"""bench.py -- images/sec of TPDM adaptive sampling, SD3-medium 1024^2 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config2|config3|config4] [--dump-outputs DIR]

The bench loads the library that build() (python -m tpdm_b200.build) left in tpdm_b200/; it compiles nothing and writes
nothing under the repository, which may be read-only where it runs.

Default workload (config2, the one the metric is quoted on): a "step" is one full adaptive trajectory for one prompt (MMDiT
forward with CFG at every denoising step, TimePredictor head, schedule update, Euler update) on synthetic text embeddings
and random-init SD3-medium weights.  With N > 1 every rank runs its own prompts (weak scaling, no data-path collective);
value = all images / max-over-ranks device time.

  value     device-resident inputs (copied to HBM before the timed region); timed with CUDA events.
  e2e       the same K trajectories through SD3PredictNextTimeStepModel.forward with HOST (pinned) embeddings/latents copied
            in every step and sigmas/final latents copied out every step.
  roofline  WHOLE denoising step: algorithmic MMDiT FLOPs x executed denoising steps / timed region, against the measured
            sustained bf16 peak (MEASURED_PEAKS.json); per-kernel figures underneath come from CUDA-event brackets that
            libtpdm_b200 records around each GEMM / attention launch of one extra trajectory (launches the device skipped
            are dropped, not credited).
  torch_eager_bf16  the bar SURVEY 8(d) names: the restated PyTorch modules in bf16 on the same GPU (cuBLASLt + SDPA), one
            denoising step, timed right after the timed regions.  A baseline leg, never the product path.
  cpu_baseline  the fp32 oracle on the host cores: ONE complete denoising step (24 blocks), x the GPU arm's measured steps.

--workload config3: BASELINE configs[2] -- 8 prompts per GPU with variable-length trajectories drained from ONE device-side
  ticket counter shared by the GPUs of the box (CUDA IPC); a step = one drain of the whole prompt list.
--workload config4: BASELINE configs[3] -- 512^2 RLOO rollout (4 prompts x 4 samples per GPU), TimePredictor fwd + bwd for
  4 PPO epochs x 2 micro-batches, one NCCL all-reduce of the flat gradient buffer per micro-batch; a step = one RLOO update.

--impl reference: the reference's own path cannot be imported offline (needs diffusers / pyrootutils / checkpoints, SURVEY
  8c), so this arm runs the fp32 oracle restatement on the host cores (kind "port").  Each bench step is a bounded sample
  that is EXECUTED, not extrapolated: `blocks_per_sample` consecutive joint blocks of the running denoising step (plus the
  step's embedders / norm_out / proj_out / TimePredictor / Euler when the slice holds them); consecutive steps continue the
  same denoising step, so K samples are K * blocks_per_sample / 24 complete denoising steps.

--dump-outputs DIR: after the timed steps, rank 0 writes what the timed path returned in its last step as DIR/<name>.npy
  (config2: the output of the last trajectory; config3: of the last drain; config4: scores, advantages and the TimePredictor
  parameters after the last update).  Inputs and weights are seeded, so two builds run with the same arguments can be
  compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec/box, SD3-M 1024^2 TPDM sampling"
UNIT = "images/s"
WORKLOAD = "SD3-medium (24 joint blocks, hidden 1536, 24 heads) random-init, 1024^2, batch 1, CFG 7.0, TPDM adaptive schedule (predict), bf16"
MAX_STEPS = 28
N_TEXT = 333
MIN_SIGMA = 0.001


def static_config(world: int) -> dict:
    """Identical in both arms (the measured quantities live at the top level of the line)."""
    return {"workload": WORKLOAD, "prompts_per_gpu_per_step": 1, "max_inference_steps": MAX_STEPS,
            "l2": "activations+weights per denoising step (~5 GB) exceed the 126 MB L2",
            "parallelism": f"prompt-sharded x{world}, no collective"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=p["bf16_tflops_sustained"], tflops_burst=p["bf16_tflops"], hbm=p["hbm_gbs"], source="measured")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# dram__bytes_read.sum + dram__bytes_write.sum per launch from one `ncu --set full` capture of round 2 (profiles/r02_attention_fast_ncu.txt;
# profiles/r02_gemm2_vs_cublas_ncu.txt: mean of the four per-block shapes 71.1 / 105.5 / 272.2 / 95.7 MB).  Algorithmic bytes per launch:
# attention 2 x 24 x 4429 x 64 x 2 B x 4 (Q, K, V, O) = 109 MB; GEMMs 71 / 136 / 237 / 128 MB.
NCU_DRAM_BYTES_PER_LAUNCH = {"gemm_bf16_tcgen05": 136.1e6, "joint_attention_tcgen05": 91.9e6}


# sm__pipe_tensor_cycles_active (% of active cycles) from the round-2 `ncu --set full` captures: the CTA-pair GEMM on the four block
# shapes (profiles/r02_gemm2_vs_cublas_ncu.txt: QKV 87, FF1 90, FF2 86, out-proj 60; FLOP-weighted over a block) and the fast attention
# kernel (profiles/r02_attention_fast_ncu.txt: 41.6, captured on the 4-softmax-warp build; the final 8-warp build is ~4 % faster)
NCU_TENSOR_PIPE_ACTIVE = {"gemm_bf16_tcgen05": (125 * 87 + 167 * 90 + 167 * 86 + 42 * 60) / 501.0, "joint_attention_tcgen05": 41.6}


def tensor_pipe_estimate(kernels: dict) -> dict:
    """Whole-step tensor-pipe activity: the ncu per-kernel percentages weighted with this run's per-kernel share of the step."""
    pct = sum(NCU_TENSOR_PIPE_ACTIVE[k] * v["share_of_trajectory"] for k, v in kernels.items() if k in NCU_TENSOR_PIPE_ACTIVE)
    return {"pct_of_step": pct, "per_kernel_pct_ncu": NCU_TENSOR_PIPE_ACTIVE,
            "how": "ncu sm__pipe_tensor_cycles_active per kernel (stand-alone captures) x share of the sampled trajectory (this run)"}


def mmdit_flops_1024() -> float:
    from oracle.sd3_oracle import mmdit_flops, sd3_medium_config

    return mmdit_flops(sd3_medium_config(), 2, 4096, N_TEXT)


def synthetic_host_inputs(seed: int, latent: int = 128, batch: int = 1):
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g).pin_memory()
    return dict(prompt_embeds=mk(batch, N_TEXT, 4096), negative_prompt_embeds=mk(batch, N_TEXT, 4096), pooled_prompt_embeds=mk(batch, 2048),
                negative_pooled_prompt_embeds=mk(batch, 2048), latents=mk(batch, 16, latent, latent))


class Dist:
    def __init__(self, world, dev):
        self.world, self.dev = world, dev

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max(self, v: float) -> float:
        if self.world == 1:
            return v
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def gather(self, v):
        if self.world == 1:
            return [v]
        out = [None] * self.world
        torch.distributed.all_gather_object(out, v)
        return out


DUMP_BYTES = 60 * 10**6      # the .npy headers stay within 64 MB as well


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each tensor as out_dir/<name>.npy, float64 as float64 and every other dtype as float32.  When the arrays exceed
    DUMP_BYTES together, each one is cut to its share of that budget: a sample of its flattened elements at fixed, seeded
    positions, the same from run to run."""
    import numpy as np

    arrays = {k: v.detach().cpu().to(torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in arrays.items()}
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        keep = max(1, t.numel() * DUMP_BYTES // total) if total > DUMP_BYTES else t.numel()
        if keep < t.numel():
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t.flatten()[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def tensors_of(out) -> dict:
    return {k: v for k, v in out.items() if torch.is_tensor(v)}


def build_model(local_rank, world, sample_size=128):
    from tpdm_b200 import _lib as L
    from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel

    lib = L.load()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)
    cfg = dict(SD3_MEDIUM_TRANSFORMER_CONFIG, sample_size=sample_size)
    return L, lib, dev, SD3PredictNextTimeStepModel, cfg


# ---------------------------------------------------------------------------------------------------------------
# config 2 (default): the metric
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    L, lib, dev, Model, cfg = build_model(local_rank, world)
    model = Model(transformer_config=cfg, torch_dtype=torch.bfloat16, device=dev)
    model.get_engine()
    D = Dist(world, dev)
    K, W = args.steps, args.warmup
    host = [synthetic_host_inputs(1000 * rank + i) for i in range(K)]
    resident = [{k: v.to(dev) for k, v in h.items()} for h in host]
    kw = dict(max_inference_steps=MAX_STEPS, guidance_scale=7.0, predict=True)

    sampler = ClockSampler(local_rank)   # started before the warm-up so that nvidia-smi's own start-up is not inside a timed region
    sampler.start()
    t_warm = time.perf_counter()
    for i in range(W):
        model(**resident[i % K], **kw)
    torch.cuda.synchronize()
    # untimed: keep the GPU under load until clocks / power have settled (the first seconds after a cold start run up to 4 %
    # slower under the 1000 W cap than the steady state; the timed regions below are exactly K steps each)
    extra = 0
    while time.perf_counter() - t_warm < 4.0 and extra < 8:
        model(**resident[extra % K], **kw)
        torch.cuda.synchronize()
        extra += 1
    D.barrier()
    sampler.rows.clear()                 # keep only the samples taken during the timed regions

    # ---- timed region 1: device-resident inputs ("value") -------------------------------------------------------
    lib.tpdm_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    e0.record()
    n_denoise = 0
    for i in range(K):
        out = model(**resident[i], **kw)
        n_denoise += out.sigmas.shape[1]
    e1.record()
    D.barrier()
    ms_value = D.max(e0.elapsed_time(e1))
    launches = int(lib.tpdm_launch_count(0))
    timed_out = out

    # ---- per-kernel sample: one more trajectory of the same workload with CUDA-event brackets around every GEMM / attention
    # / LayerNorm / adaLN launch (kept out of region 1: ~250 extra event records per denoising step perturb it by a few %)
    L.check(lib.tpdm_profile_start(8192))
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    prof_out = model(**resident[0], **kw)
    p1.record()
    torch.cuda.synchronize()
    ms_prof, prof_steps = p0.elapsed_time(p1), prof_out.sigmas.shape[1]
    pms, pfl, pct = (C.c_double * 4)(), (C.c_double * 4)(), (C.c_longlong * 4)()
    L.check(lib.tpdm_profile_stop(pms, pfl, pct, 4))
    dropped = int(lib.tpdm_profile_dropped())

    # ---- timed region 2: host buffers through the public API ("e2e") --------------------------------------------
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    d2h = 0
    D.barrier()
    e0.record()
    for i in range(K):
        out = model(**{k: v.to(dev, non_blocking=True) for k, v in host[i].items()}, **kw)
        res = (out.latents.cpu(), out.sigmas.cpu(), out.alphas.cpu(), out.betas.cpu(), out.logprobs.cpu())
        d2h = sum(t.numel() * t.element_size() for t in res)
    e1.record()
    D.barrier()
    ms_e2e = D.max(e0.elapsed_time(e1))
    clocks = sampler.stop()

    # ---- outside every timed region: the step after the path, VAE decode of one final latent to 1024^2 uint8 pixels
    vae_ms = None
    try:
        from tpdm_b200.vae import AutoencoderKL

        vae = AutoencoderKL(device=dev, dtype=torch.float32)
        lat = out.latents.float()
        vae.decode_latents(lat, "uint8")
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        v0.record()
        for _ in range(3):
            vae.decode_latents(lat, "uint8")
        v1.record()
        torch.cuda.synchronize()
        vae_ms = v0.elapsed_time(v1) / 3
        del vae
    except Exception as e:  # the decode is not part of the metric: report, do not fail the bench
        vae_ms = f"failed: {e}"

    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tensors_of(timed_out))
    eager = torch_eager_bf16_step(dev) if world == 1 else None
    pk = peaks()
    steps_per_image = n_denoise / K
    ms_per_denoise = ms_value / n_denoise
    flop_step = mmdit_flops_1024()
    step_tflops = flop_step / (ms_per_denoise / 1e3) / 1e12
    kernels = {}
    for idx, name in enumerate(("gemm_bf16_tcgen05", "joint_attention_tcgen05")):
        if pct[idx]:
            tf = pfl[idx] / pms[idx] / 1e9
            kernels[name] = dict(ms_total=pms[idx], launches=int(pct[idx]), tflops=tf, frac=tf / pk["tflops"], share_of_trajectory=pms[idx] / ms_prof,
                                 ms_per_denoise_step=pms[idx] / prof_steps, dram_bytes_per_launch_ncu=NCU_DRAM_BYTES_PER_LAUNCH.get(name))
    hbm = {}
    for idx, name in ((2, "ln_modulate"), (3, "adaln_gemv_bf16")):
        if pct[idx]:
            gbs = pfl[idx] / pms[idx] / 1e6
            hbm[name] = dict(ms_total=pms[idx], launches=int(pct[idx]), gb_per_s=gbs, frac_of_hbm_peak=gbs / float(pk["hbm"]),
                             share_of_trajectory=pms[idx] / ms_prof)
    dom = max(kernels, key=lambda k: kernels[k]["ms_total"]) if kernels else None
    roofline = dict(
        bound="tensor", scope="whole denoising step (all kernels, launch gaps included)", achieved=step_tflops, peak=pk["tflops"], unit="TFLOP/s",
        frac=step_tflops / pk["tflops"], frac_of_burst_peak=step_tflops / pk["tflops_burst"], peak_source=pk["source"] + " (sustained bf16)",
        algorithmic_tflop_per_denoise_step=flop_step / 1e12, dominant_kernel=dom, traffic=NCU_DRAM_BYTES_PER_LAUNCH.get(dom),
        traffic_source="profiles/: dram__bytes_read+write per launch of the dominant kernel, ncu --set full",
        kernels=kernels, hbm_kernels=hbm, kernel_time_share_of_trajectory=sum(k["share_of_trajectory"] for k in list(kernels.values()) + list(hbm.values())),
        sampled_over=f"one extra trajectory ({prof_steps} denoising steps) with per-launch CUDA events; {dropped} launches of the speculatively "
                     "enqueued last step were skipped on the device and are not credited",
        kernel_time_share_note="the share sums the FOUR bracketed kernel classes only (GEMM, attention, LayerNorm-modulate, adaLN GEMV); the other "
                               "~14 small kernels of a step are 1.5 % of its kernel time in the ncu launch list (profiles/r02_launch_shares*.txt), and "
                               "the event brackets themselves break programmatic-dependent-launch overlap in this sampled trajectory",
        tensor_pipe_active_estimate=tensor_pipe_estimate(kernels),
        tensor_pipe_note="sm__pipe_tensor_cycles_active per kernel: profiles/ (ncu); this line reports algorithmic FLOP/s over the sustained peak")
    line = {
        "metric": METRIC, "value": world * K / (ms_value / 1e3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_value / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (N(0,1) text embeddings and latents; random-init SD3-medium + TPM weights)",
        "config": static_config(world), "denoise_steps_per_image": steps_per_image, "untimed_settle_images_after_warmup": extra,
        "e2e": {"value": world * K / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
        "mmdit_step": {"ms_per_denoise_step": ms_per_denoise, "tflops": step_tflops, "frac_of_sustained_peak": step_tflops / pk["tflops"]},
    }
    if eager is not None:
        eager["images_per_s"] = 1e3 / (eager["ms_per_denoise_step"] * steps_per_image) if "ms_per_denoise_step" in eager else None
        if eager.get("images_per_s"):
            eager["ours_over_eager"] = line["value"] / eager["images_per_s"]
        line["torch_eager_bf16"] = eager
    if isinstance(vae_ms, float):
        line["vae_decode"] = {"ms_per_image": vae_ms, "tflops": 10.472e12 / vae_ms / 1e9, "in_timed_region": False,
                              "images_per_s_with_decode": world / (ms_value / K / 1e3 + vae_ms / 1e3),
                              "note": "SD3 VAE decoder, 128x128 latent -> 1024^2 uint8, measured after the timed regions"}
    else:
        line["vae_decode"] = {"error": str(vae_ms)}
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(steps_per_image)
    return line


def torch_eager_bf16_step(dev):
    """SURVEY 8(d): 'PyTorch-eager bf16 on the same B200 (cuBLASLt + SDPA)' -- what the reference would execute.  The restated
    modules (oracle/, the reference's own classes need diffusers) are cast to bf16 and run one denoising step under torch
    eager: MMDiT forward with CFG (Bt = 2), CFG combines, TimePredictor, Euler.  Baseline leg only."""
    try:
        from oracle import sd3_oracle as O

        torch.manual_seed(1234)
        pipe = O.OraclePipeline(O.sd3_medium_config()).to(device=dev, dtype=torch.bfloat16)
        g = torch.Generator(device=dev).manual_seed(0)
        mk = lambda *s: torch.randn(*s, device=dev, generator=g, dtype=torch.bfloat16)
        lat, enc, pooled = mk(1, 16, 128, 128), mk(2, N_TEXT, 4096), mk(2, 2048)
        sigma = torch.full((1,), 0.7, device=dev, dtype=torch.bfloat16)

        def step():
            with torch.no_grad():
                v, temb, h1, h2 = pipe.transformer(torch.cat([lat] * 2), enc, pooled, sigma.repeat(2) * 1000)
                vu, vt = v.chunk(2)
                v = vu + 7.0 * (vt - vu)
                tu, tt = temb.chunk(2)
                temb = tu + 7.0 * (tt - tu)
                h1u, h1t = h1.chunk(2)
                h1 = h1u + 7.0 * (h1t - h1u)
                h2u, h2t = h2.chunk(2)
                h2 = h2u + 7.0 * (h2t - h2u)
                hc = torch.cat([O.reshape_hidden_states_to_2d(h1, 64, 64), O.reshape_hidden_states_to_2d(h2, 64, 64)], dim=1)
                ab = pipe.time_predictor(hc, temb)
                ratio = (ab[:, 0] - 1) / (ab[:, 0] + ab[:, 1] - 2)
                return O.custom_step(v, sigma * ratio, sigma, lat)

        backend = "default dispatch"
        ctx = None
        try:
            from torch.nn.attention import SDPBackend, sdpa_kernel

            ctx = lambda: sdpa_kernel([SDPBackend.CUDNN_ATTENTION, SDPBackend.FLASH_ATTENTION], set_priority=True)
            with ctx():
                step()
            backend = "cuDNN attention preferred, flash fallback"
        except Exception:
            ctx = None
        import contextlib

        cm = ctx if ctx is not None else contextlib.nullcontext
        with cm():
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = 5
            for _ in range(n):
                step()
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        del pipe
        torch.cuda.empty_cache()
        return {"ms_per_denoise_step": ms, "tflops": mmdit_flops_1024() / ms / 1e9, "sdpa_backend": backend,
                "what": "restated PyTorch modules in bf16, torch eager (cuBLASLt GEMMs + SDPA), one denoising step with CFG, mean of 5 after 2 warm-ups",
                "in_timed_region": False}
    except Exception as e:   # a baseline leg must never fail the bench
        return {"error": str(e).splitlines()[0][:200]}


# ---------------------------------------------------------------------------------------------------------------
# host-CPU legs: the fp32 oracle
# ---------------------------------------------------------------------------------------------------------------
class OracleStepRunner:
    """One 1024^2 denoising step of the fp32 oracle with CFG (Bt = 2), executable in slices of consecutive joint blocks."""

    def __init__(self):
        from oracle import sd3_oracle as O

        self.O = O
        torch.set_num_threads(os.cpu_count())
        torch.manual_seed(0)
        self.pipe = O.OraclePipeline(O.sd3_medium_config())
        g = torch.Generator().manual_seed(0)
        self.enc, self.pooled = torch.randn(2, N_TEXT, 4096, generator=g), torch.randn(2, 2048, generator=g)
        self.lat = torch.randn(1, 16, 128, 128, generator=g)
        self.sigma = torch.ones(1)
        self.block = 0
        self.ratio = None
        self.steps_done = 0

    @torch.no_grad()
    def run_blocks(self, n: int) -> None:
        """Executes the next n joint blocks of the running denoising step (wrapping into the next step)."""
        tr = self.pipe.transformer
        L = len(tr.transformer_blocks)
        for _ in range(n):
            if self.block == 0:
                lat2 = torch.cat([self.lat] * 2)
                self.hs = tr.pos_embed(lat2)
                self.h1 = self.hs.clone()
                self.temb = tr.time_text_embed(self.sigma.repeat(2) * 1000, self.pooled)
                self.ctx = tr.context_embedder(self.enc)
            self.ctx, self.hs = tr.transformer_blocks[self.block](self.hs, self.ctx, self.temb)
            self.block += 1
            if self.block == L:
                self._tail()
                self.block = 0

    def _tail(self):
        O, tr = self.O, self.pipe.transformer
        h2 = tr.norm_out(self.hs, self.temb)
        v = tr.unpatchify(tr.proj_out(h2), 128, 128) if hasattr(tr, "unpatchify") else None
        if v is None:   # restated inline: Linear D -> 64, nhwpqc -> nchpwq (transformer_sd3.py:374-399)
            o = tr.proj_out(h2).reshape(2, 64, 64, 2, 2, 16)
            v = torch.einsum("nhwpqc->nchpwq", o).reshape(2, 16, 128, 128)
        vu, vt = v.chunk(2)
        v = vu + 7.0 * (vt - vu)
        tu, tt = self.temb.chunk(2)
        temb = tu + 7.0 * (tt - tu)
        h1u, h1t = self.h1.chunk(2)
        h1 = h1u + 7.0 * (h1t - h1u)
        h2u, h2t = h2.chunk(2)
        h2c = h2u + 7.0 * (h2t - h2u)
        hc = torch.cat([O.reshape_hidden_states_to_2d(h1, 64, 64), O.reshape_hidden_states_to_2d(h2c, 64, 64)], dim=1)
        ab = self.pipe.time_predictor(hc, temb)
        self.ratio = float(((ab[:, 0] - 1) / (ab[:, 0] + ab[:, 1] - 2)).clamp(1e-3, 0.999))
        sigma_next = self.sigma * self.ratio
        self.lat = O.custom_step(v, sigma_next, self.sigma, self.lat)
        self.sigma = sigma_next if float(sigma_next) >= MIN_SIGMA else torch.ones(1)     # next image
        self.steps_done += 1


def steps_from_ratio(ratio: float) -> int:
    """Denoising steps until sigma_next = ratio^k < min_sigma with a constant ratio (the reference init is bias dominated:
    the GPU arm measures 22-23)."""
    return int(math.floor(math.log(MIN_SIGMA) / math.log(ratio))) + 1


def cpu_baseline(steps_per_image: float):
    """ONE complete denoising step (embedders, 24 joint blocks, norm_out / proj_out, TimePredictor, Euler) of the fp32 oracle on
    all host cores, timed; images/s = 1 / (step time x the GPU arm's measured denoising steps per image)."""
    r = OracleStepRunner()
    t0 = time.perf_counter()
    r.run_blocks(24)
    step_s = time.perf_counter() - t0
    return {"value": 1.0 / (step_s * steps_per_image), "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"fp32 oracle, ONE complete 1024^2 denoising step with CFG (Bt=2, 24 joint blocks + embedders + tail + TPM + Euler) = "
                      f"{step_s:.1f} s, x {steps_per_image:.2f} denoising steps per image measured by the GPU arm",
            "step_seconds": step_s}


def run_reference(args, rank, world):
    if rank != 0:
        return None
    K, W = args.steps, args.warmup
    r = OracleStepRunner()
    # size the sample: one untimed block tells how many of the 24 blocks fit a ~210 s run of K + W samples
    t0 = time.perf_counter()
    r.run_blocks(1)
    t_block = time.perf_counter() - t0
    per_sample_s = 210.0 / max(1, K + W)
    nb = 24
    for cand in (24, 12, 8, 6, 4, 3, 2, 1):
        nb = cand
        if cand * t_block <= per_sample_s:
            break
    r.run_blocks(24 - 1)                      # finish the step that the sizing block started (untimed)
    for _ in range(W):
        r.run_blocks(nb)
    while r.block != 0:                       # timed samples start at a step boundary
        r.run_blocks(1)
    done_before = r.steps_done
    t0 = time.perf_counter()
    for _ in range(K):
        r.run_blocks(nb)
    total_s = time.perf_counter() - t0
    denoise_steps = K * nb / 24.0
    steps_per_image = steps_from_ratio(r.ratio) if r.ratio else 23
    v = denoise_steps / steps_per_image / total_s
    cb = {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
          "sample": f"fp32 oracle on all host cores; each bench step EXECUTES {nb} consecutive joint blocks of the running 1024^2 denoising step "
                    f"(+ embedders / tail / TPM / Euler when the slice holds them): {K} samples = {denoise_steps:.2f} complete denoising steps in "
                    f"{total_s:.1f} s ({r.steps_done - done_before} step tails executed); x {steps_per_image} denoising steps per image from the "
                    f"oracle's own TimePredictor (Beta mode {r.ratio:.4f})",
          "blocks_per_sample": nb, "seconds_per_denoise_step": total_s / denoise_steps}
    return {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_s / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (N(0,1) text embeddings and latents; random-init SD3-medium + TPM weights)",
            "config": static_config(world), "denoise_steps_per_image": steps_per_image, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "host CPU only; rank 0 runs, other ranks exit"}


# ---------------------------------------------------------------------------------------------------------------
# config 3: variable-length trajectories, one device-side queue for the whole box
# ---------------------------------------------------------------------------------------------------------------
def run_config3(args, rank, world, local_rank):
    from tpdm_b200.work_queue import SharedTicket

    L, lib, dev, Model, cfg = build_model(local_rank, world)
    model = Model(transformer_config=cfg, torch_dtype=torch.bfloat16, device=dev, init_alpha=1.5, init_beta=0.5)
    with torch.no_grad():       # (alpha, beta) depend on the hidden states: 6..28 step trajectories (SURVEY 8d cfg 3)
        tp = model.time_predictor
        tp.fc2.weight.mul_(4.0)
        tp.fc1.weight.mul_(4.0)
        tp.conv2.weight.mul_(2.0)
    model.get_engine()
    D = Dist(world, dev)
    K, W, slots = args.steps, args.warmup, args.slots
    P = args.prompts_per_gpu * world

    def inputs(i):
        g = torch.Generator().manual_seed(5000 + i)
        mk = lambda *s: torch.randn(*s, generator=g).to(dev)
        return dict(prompt_embeds=mk(1, N_TEXT, 4096), negative_prompt_embeds=mk(1, N_TEXT, 4096), pooled_prompt_embeds=mk(1, 2048),
                    negative_pooled_prompt_embeds=mk(1, 2048), latents=mk(1, 16, 128, 128))

    allin = [inputs(i) for i in range(P)]      # every GPU holds every prompt: whoever draws the ticket runs it
    cat = {k: torch.cat([a[k] for a in allin]) for k in allin[0]}
    del allin
    ticket = SharedTicket.create()

    def drain(order_mode):
        ticket.reset()
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = model.sample_queue(cat["prompt_embeds"], cat["negative_prompt_embeds"], cat["pooled_prompt_embeds"],
                                 cat["negative_pooled_prompt_embeds"], latents=cat["latents"], slots=slots, max_inference_steps=MAX_STEPS,
                                 ticket=ticket, schedule=order_mode)
        e1.record()
        torch.cuda.synchronize()
        return out, e0.elapsed_time(e1)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(W):
        drain(args.schedule)
    D.barrier()
    sampler.rows.clear()
    lib.tpdm_launch_count(1)
    ms_total, busy, dsteps, out = 0.0, [], [], None
    for _ in range(K):
        out, ms = drain(args.schedule)
        mk = D.max(ms)
        ms_total += mk
        busy.append(ms / mk)
        dsteps.append(int(out.device_steps))
    launches = int(lib.tpdm_launch_count(0))
    clocks = sampler.stop()
    steps = out.steps.clone()
    if world > 1:
        torch.distributed.all_reduce(steps)
    busy_all, dsteps_all = D.gather(sum(busy) / len(busy)), D.gather(dsteps[-1])
    mine = D.gather(int((out.steps > 0).sum()))
    # single-slot step time on this GPU = the unit of the lower bound
    one = {k: v[:1] for k, v in cat.items()}
    o1 = model(**one, max_inference_steps=MAX_STEPS, predict=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    o1 = model(**one, max_inference_steps=MAX_STEPS, predict=True)
    e1.record()
    torch.cuda.synchronize()
    ms_step1 = e0.elapsed_time(e1) / o1.sigmas.shape[1]
    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tensors_of(out))
    st = steps.tolist()
    assert all(s > 0 for s in st), "a prompt was not processed"
    assert sum(mine) == P, "a prompt was processed twice"
    makespan = ms_total / K
    hist = {}
    for s_ in st:
        hist[s_] = hist.get(s_, 0) + 1
    bound_ms = sum(st) * ms_step1 / world
    return {
        "metric": "images/sec/box, SD3-M 1024^2 TPDM sampling, variable-length trajectories (BASELINE configs[2])", "value": P / (makespan / 1e3),
        "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": makespan, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic; TimePredictor fc/conv2 weights scaled so that alpha/beta depend on the hidden states",
        "config": {"workload": f"SD3-medium 1024^2, {P} prompts ({args.prompts_per_gpu} per GPU) of different trajectory length drained from one "
                               f"device-side ticket counter shared by {world} GPU(s) (CUDA IPC), {slots} in-flight slots per GPU, schedule={args.schedule}",
                   "parallelism": f"prompt queue x{world}, no collective"},
        "total_denoise_steps": sum(st), "steps_histogram": dict(sorted(hist.items())), "prompts_per_gpu": mine, "device_steps_per_gpu": dsteps_all,
        "busy_fraction_per_gpu": busy_all, "single_slot_ms_per_denoise_step": ms_step1,
        "lower_bound_ms": bound_ms, "efficiency_vs_sum_steps_over_n_bound": bound_ms / makespan,
        "gpu_launches": launches, "clocks": clocks,
        "e2e": {"value": P / (makespan / 1e3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "prompts are resident on every GPU before the drain (that is what lets any GPU take any ticket)"},
    }


# ---------------------------------------------------------------------------------------------------------------
# config 4: RLOO rollout + TimePredictor update with the gradient all-reduce
# ---------------------------------------------------------------------------------------------------------------
def run_config4(args, rank, world, local_rank):
    import torch.distributed as dist

    L, lib, dev, Model, cfg = build_model(local_rank, world, sample_size=64)
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModelRLOOWrapper
    from tpdm_b200.rloo import rloo_update
    from tpdm_b200.tpm_training import TimePredictorTrainer

    torch.manual_seed(1234)
    wrapper = SD3PredictNextTimeStepModelRLOOWrapper(transformer_config=cfg, torch_dtype=torch.bfloat16, device=dev, min_sigma=0.01,
                                                     init_alpha=2.5, init_beta=1.0, max_inference_steps=MAX_STEPS)   # launch_sd3_train.sh:16-19
    agent = wrapper.agent_model
    agent.get_engine()
    D = Dist(world, dev)
    K, W, rloo_k, prompts, mbs = args.steps, args.warmup, 4, 4, 8
    trainer = TimePredictorTrainer(agent.time_predictor, grid=32, max_samples=mbs * MAX_STEPS, lr=1e-6, betas=(0.9, 0.99), eps=1e-5)
    gen = torch.Generator().manual_seed(1234 + rank * 100003)          # rloo_trainer.py:133
    g = torch.Generator().manual_seed(77 + rank)
    mk = lambda *s: torch.randn(*s, generator=g).to(dev)
    data = dict(prompt_embeds=mk(prompts, N_TEXT, 4096), negative_prompt_embeds=mk(prompts, N_TEXT, 4096), pooled_prompt_embeds=mk(prompts, 2048),
                negative_pooled_prompt_embeds=mk(prompts, 2048))
    reward = lambda latents, outputs: -(latents.float() ** 2).mean(dim=(1, 2, 3))       # synthetic reward (SURVEY 8d cfg 4)

    def update():
        return rloo_update(wrapper, trainer, data, reward, rloo_k=rloo_k, num_ppo_epochs=4, micro_batch_size=mbs, cliprange=0.2, gamma=0.97,
                           generator=gen)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(W):
        update()
    D.barrier()
    sampler.rows.clear()
    lib.tpdm_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    e0.record()
    steps_avg, last = [], None
    for _ in range(K):
        last = update()
        steps_avg.append(last["steps"])
    e1.record()
    D.barrier()
    ms = D.max(e0.elapsed_time(e1))
    launches = int(lib.tpdm_launch_count(0))
    clocks = sampler.stop()
    # correctness of the exchange, outside the timed region: all-reduced buffer == sum of the per-rank buffers; parameters identical
    check = "single GPU: no exchange"
    if world > 1:
        outputs = wrapper.sample({**wrapper.rloo_repeat(dict(data), rloo_k), "predict": False, "generator": gen})
        x = outputs["hidden_states_combineds"].permute(0, 1, 3, 4, 2)
        idx = torch.arange(mbs, device=dev)
        adv = torch.linspace(-1.0, 1.0, mbs, device=dev) * (1 + rank)
        mb_args = (outputs["sigmas"][idx], outputs["logprobs"][idx], x[idx], outputs["tembs"][idx], adv)
        mb_kw = dict(min_sigma=agent.min_sigma, optimizer_step=False)
        trainer.ppo_update(*mb_args, **mb_kw, all_reduce=False)
        local = trainer.reduce_buf.clone()
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        trainer.ppo_update(*mb_args, **mb_kw)                       # the product path: ONE all-reduce of gradients + loss + NaN flag
        red = trainer.reduce_buf.clone()
        err = float((torch.stack(gathered).sum(0) - red).norm() / red.norm())      # float atomics in the backward reorder sums
        ref = trainer.params.clone()
        dist.broadcast(ref, 0)
        same = bool(torch.equal(ref, trainer.params))
        flags = D.gather((err, same))
        assert all(f[0] < 1e-3 and f[1] for f in flags), flags
        check = (f"all-reduced gradient+loss buffer == sum of the {world} per-rank buffers (rel err {max(f[0] for f in flags):.1e}); "
                 f"parameters bit-identical on all ranks after {K + W} updates")
    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(scores=last["scores"], advantages=last["advantages"], tpm_params=trainer.params))
    rollouts = prompts * rloo_k
    return {
        "metric": "rollouts/sec/box, SD3-M 512^2 RLOO update (BASELINE configs[3])", "value": world * K * rollouts / (ms / 1e3), "unit": "rollouts/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic embeddings, device-side Beta draws, synthetic reward -mean(latent^2)",
        "config": {"workload": f"SD3-medium 512^2 RLOO: {prompts} prompts x rloo_k {rloo_k} = {rollouts} rollouts per GPU (transformer batch {2 * rollouts}), "
                               f"4 PPO epochs x {rollouts // mbs} micro-batches of {mbs}: TimePredictor fwd+bwd, one NCCL all-reduce of the flat "
                               f"{trainer.reduce_buf.numel() * 4 / 1e6:.1f} MB gradient+loss buffer per micro-batch, fused clip+AdamW",
                   "parallelism": f"data parallel x{world}, all-reduce of TPM gradients only"},
        "mean_denoise_steps_per_rollout": sum(steps_avg) / len(steps_avg), "last_update": last["logs"][-1], "allreduce_check": check,
        "allreduce_bytes": trainer.reduce_buf.numel() * 4, "gpu_launches": launches, "clocks": clocks,
        "e2e": {"value": world * K * rollouts / (ms / 1e3), "unit": "rollouts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": rollouts * 4,
                "note": "an update reads the scores back (B floats); embeddings are resident as in the reference's pre_process mode"},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config4"])
    ap.add_argument("--slots", type=int, default=2, help="config3: prompts in flight per GPU")
    ap.add_argument("--prompts-per-gpu", type=int, default=8, help="config3")
    ap.add_argument("--schedule", default="fifo", choices=["fifo", "lpt"], help="config3: ticket order (lpt: longest expected trajectory first)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"config2": 8, "config3": 2, "config4": 2}[args.workload]
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        fn = {"config2": run_ours, "config3": run_config3, "config4": run_config4}[args.workload]
        line = fn(args, rank, world, local_rank)
        if line is not None:
            print(json.dumps(line), flush=True)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
