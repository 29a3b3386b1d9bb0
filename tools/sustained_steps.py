"""Denoising steps of the SD3-medium 1024^2 trajectory back to back for a few seconds, under the power cap: ms per step with the
median SM clock and power.  Stand-alone kernel timings (short, cool, full clocks) do not predict the trajectory on a power-capped
B200 -- a kernel that is faster but draws more power lowers the clock of everything else -- so kernel variants are compared with
this loop:   TPDM_B200_LIB=tpdm_b200/_build/libtpdm_<variant>.so python tools/sustained_steps.py [seconds]"""
import os
import subprocess
import sys
import threading
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tpdm_b200 import _lib as _L  # noqa: E402
from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel  # noqa: E402

seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 8.0
torch.manual_seed(1234)
model = SD3PredictNextTimeStepModel(transformer_config=SD3_MEDIUM_TRANSFORMER_CONFIG, torch_dtype=torch.bfloat16, device="cuda")
g = torch.Generator().manual_seed(0)
mk = lambda *s: torch.randn(*s, generator=g).cuda()
kw = dict(prompt_embeds=mk(1, 333, 4096), negative_prompt_embeds=mk(1, 333, 4096), pooled_prompt_embeds=mk(1, 2048),
          negative_pooled_prompt_embeds=mk(1, 2048), latents=mk(1, 16, 128, 128))
for _ in range(2):
    out = model(**kw, max_inference_steps=28, predict=True)
torch.cuda.synchronize()
samples, stop = [], [False]


def sample():
    while not stop[0]:
        r = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits"], capture_output=True, text=True)
        try:
            c, pw = r.stdout.strip().split(",")
            samples.append((float(c), float(pw)))
        except Exception:
            pass
        time.sleep(0.25)


th = threading.Thread(target=sample, daemon=True)
th.start()
e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
steps, images, t0 = 0, 0, time.perf_counter()
e0.record()
while time.perf_counter() - t0 < seconds:
    out = model(**kw, max_inference_steps=28, predict=True)
    steps += int(out.sigmas.shape[1]) - 1
    images += 1
e1.record()
torch.cuda.synchronize()
stop[0] = True
ms = e0.elapsed_time(e1)
clk = sorted(s[0] for s in samples)
pw = sorted(s[1] for s in samples)
print(f"{os.environ.get('TPDM_B200_LIB', 'product')}: {images} images, {steps} steps, "
      f"{ms / steps:.3f} ms per denoising step, {images / ms * 1e3:.3f} images/s; median SM clock {clk[len(clk) // 2]:.0f} MHz, "
      f"median power {pw[len(pw) // 2]:.0f} W; attention CTAs that took the exact pass: {_L.load().tpdm_attention_redo_total()}", flush=True)
