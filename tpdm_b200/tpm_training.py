"""Training half of the TPDM path (SURVEY.md section 8a rows R1-R3) on top of libtpdm_b200.so: TimePredictor replay with
gradients, PPO-clip loss on summed log-probs, one flat-buffer gradient all-reduce over NCCL and a fused clip + AdamW
step.  Mirrors what CommonRLOOTrainer does for one micro-batch (/root/reference/src/train/rloo_trainer.py:485-523) for
the only trainable module, the TimePredictor (modeling_sd3_pnt.py:760-763)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import _lib as L

NAMES = ("conv1.weight", "conv1.bias", "norm1.linear.weight", "norm1.linear.bias", "norm1.norm.weight", "norm1.norm.bias",
         "conv2.weight", "conv2.bias", "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")


def _to_packed(name: str, t: torch.Tensor) -> torch.Tensor:
    if name == "conv1.weight":   # [C1, 2D, 3, 3] -> [C1, 9, 2D]
        return t.permute(0, 2, 3, 1).reshape(-1)
    if name == "conv2.weight":   # [oc, c, 3, 3] -> [9, c, oc]
        return t.permute(2, 3, 1, 0).reshape(-1)
    return t.reshape(-1)


def _from_packed(name: str, flat: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    if name == "conv1.weight":
        c1, c_in = like.shape[0], like.shape[1]
        return flat.reshape(c1, 3, 3, c_in).permute(0, 3, 1, 2)
    if name == "conv2.weight":
        oc, c = like.shape[0], like.shape[1]
        return flat.reshape(3, 3, c, oc).permute(3, 2, 0, 1)
    return flat.reshape(like.shape)


class TimePredictorTrainer:
    """Owns the flat fp32 master copy of the TimePredictor parameters, their gradients and the AdamW state."""

    def __init__(self, time_predictor, grid: int, max_samples: int, lr: float = 1e-6, betas=(0.9, 0.99), eps: float = 1e-5,
                 weight_decay: float = 0.0, max_grad_norm: float = 1.0):
        lib = L.load()
        self.module = time_predictor
        sd = time_predictor.state_dict()
        dev = sd["fc2.weight"].device
        if dev.type != "cuda":
            raise RuntimeError("TimePredictorTrainer runs on CUDA only (no CPU path)")
        self.device, self.g, self.max_samples = dev, grid, max_samples
        self.C1 = sd["conv1.weight"].shape[0]
        self.D = sd["conv1.weight"].shape[1] // 2
        self.lr, self.betas, self.eps, self.weight_decay, self.max_grad_norm = lr, betas, eps, weight_decay, max_grad_norm
        off = (C.c_longlong * 13)()
        L.check(lib.tpdm_tpm_param_offsets(self.D, self.C1, off))
        self.off = list(off)
        n = self.off[12]
        self.params = torch.zeros(n, device=dev, dtype=torch.float32)
        # ONE buffer goes through the data-parallel all-reduce: the gradients followed by {loss, non-finite-loss flag}
        # (rloo_trainer.py:497-501: gather(loss) + NaN guard + backward become one exchange; SURVEY 2.3 C3 + C4)
        self.reduce_buf = torch.zeros(n + 2, device=dev, dtype=torch.float32)
        self.grads = self.reduce_buf[:n]
        self.tail = self.reduce_buf[n:]
        self.m, self.v = torch.zeros_like(self.params), torch.zeros_like(self.params)
        self.sumsq = torch.zeros(1, device=dev, dtype=torch.float64)
        self.n_conv1 = sd["conv1.weight"].numel()
        self.conv1_bf16 = torch.zeros(self.n_conv1, device=dev, dtype=torch.bfloat16)
        self.load_from_module()
        with torch.cuda.device(dev):
            nbytes = lib.tpdm_tpm_trainer_workspace_bytes(self.D, self.C1, grid, max_samples)
            self.workspace, base = L.aligned_workspace(nbytes, dev)
            h = L.vp()
            L.check(lib.tpdm_tpm_trainer_create(self.D, self.C1, grid, max_samples, float(time_predictor.epsilon), base, nbytes, C.byref(h)))
            self.handle = h
            L.check(lib.tpdm_tpm_trainer_bind(h, L.ptr(self.params), L.ptr(self.grads), L.ptr(self.conv1_bf16)))
        self.step_count = 0
        self._keep = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                L.load().tpdm_tpm_trainer_destroy(self.handle)
        except Exception:
            pass

    # ---- parameter hand-over -------------------------------------------------------------------------------------
    def load_from_module(self):
        sd = self.module.state_dict()
        for i, name in enumerate(NAMES):
            flat = _to_packed(name, sd[name].detach().to(device=self.device, dtype=torch.float32))
            self.params[self.off[i]: self.off[i] + flat.numel()].copy_(flat)
        self.conv1_bf16.copy_(self.params[: self.n_conv1])

    def tensors(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        sd = self.module.state_dict()
        return {name: _from_packed(name, flat[self.off[i]: self.off[i] + sd[name].numel()], sd[name]) for i, name in enumerate(NAMES)}

    def sync_to_module(self):
        """Write the fp32 master parameters back into the nn.Module (PyTorch layouts, module dtype)."""
        new = self.tensors(self.params)
        with torch.no_grad():
            for name, p in self.module.state_dict().items():
                p.copy_(new[name])

    def grad_dict(self) -> Dict[str, torch.Tensor]:
        return {k: v.clone() for k, v in self.tensors(self.grads).items()}

    # ---- forward / backward ----------------------------------------------------------------------------------------
    def forward(self, x_nhwc: torch.Tensor, temb: torch.Tensor) -> torch.Tensor:
        """x_nhwc: (ns, g, g, 2D) bf16 contiguous (or any view whose storage is NHWC-contiguous); temb: (ns, D)."""
        lib = L.load()
        ns = x_nhwc.shape[0]
        x = x_nhwc.to(torch.bfloat16).contiguous()
        t = temb.to(device=self.device, dtype=torch.float32).contiguous()
        if x.shape != (ns, self.g, self.g, 2 * self.D) or t.shape != (ns, self.D):
            raise ValueError(f"expected x (ns,{self.g},{self.g},{2 * self.D}) and temb (ns,{self.D}); got {tuple(x.shape)}, {tuple(t.shape)}")
        self._keep = (x, t)   # borrowed by the library until backward() has run
        self._generation = getattr(self, "_generation", 0) + 1   # the saved activations belong to THIS forward
        ab = torch.empty(ns, 2, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            L.check(lib.tpdm_tpm_train_forward(self.handle, L.ptr(x), L.ptr(t), ns, L.ptr(ab), L.stream_ptr()))
        return ab

    def backward(self, dz: torch.Tensor) -> None:
        lib = L.load()
        d = dz.to(device=self.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(self.device):
            L.check(lib.tpdm_tpm_train_backward(self.handle, L.ptr(d), L.stream_ptr()))

    # ---- one micro-batch of rloo_trainer.py:485-523 ------------------------------------------------------------------
    def ppo_update(self, sigmas: torch.Tensor, old_logprobs: torch.Tensor, tpm_inputs_nhwc: torch.Tensor, tembs: torch.Tensor,
                   advantages: torch.Tensor, min_sigma: float, cliprange: float = 0.2, epsilon: float = 1e-3, relative: bool = True,
                   optimizer_step: bool = True, prediction_type: str = "alpha_beta", all_reduce: bool = True) -> Dict[str, torch.Tensor]:
        """sigmas / old_logprobs (mb, T); tpm_inputs_nhwc (mb, T, g, g, 2D) bf16; tembs (mb, T, D); advantages (mb,).
        Returns device scalars: loss (mean over ranks), clipfrac, approxkl, ratio, nonfinite (how many ranks saw a NaN / Inf
        loss: > 0 means the optimizer step was skipped on EVERY rank) and, with optimizer_step, grad_norm."""
        if prediction_type not in ("alpha_beta", "mode_concentration"):
            raise ValueError(f"unknown prediction_type {prediction_type!r}")
        lib = L.load()
        mb, T = sigmas.shape
        f32 = dict(device=self.device, dtype=torch.float32)
        ab = self.forward(tpm_inputs_nhwc.reshape(mb * T, self.g, self.g, 2 * self.D), tembs.reshape(mb * T, self.D))
        sig, old, adv = sigmas.to(**f32).contiguous(), old_logprobs.to(**f32).contiguous(), advantages.to(**f32).contiguous()
        new_lp = torch.empty(mb, T, **f32)
        dz = torch.empty(mb * T, 2, **f32)
        stats = torch.empty(4, **f32)
        with torch.cuda.device(self.device):
            L.check(lib.tpdm_ppo_clip_loss(L.ptr(ab), L.ptr(sig), L.ptr(old), L.ptr(adv), mb, T, float(min_sigma), float(epsilon),
                                           1 if relative else 0, 0 if prediction_type == "alpha_beta" else 1, float(cliprange),
                                           float(self.module.epsilon), L.ptr(new_lp), L.ptr(dz), L.ptr(stats), self.tail.data_ptr(),
                                           L.stream_ptr()))
        self.backward(dz)      # overwrites self.grads; the tail written above sits right behind them
        world = dist.get_world_size() if dist.is_initialized() else 1
        if not all_reduce:      # local gradient only (tests of the exchange itself)
            world = 1
        if world > 1:   # the only exchange step of the path: TPM gradients + loss + NaN flag in ONE buffer (rloo_trainer.py:497-501)
            dist.all_reduce(self.reduce_buf, op=dist.ReduceOp.SUM)
        out = dict(loss=self.tail[0] / world, local_loss=stats[0], clipfrac=stats[1], approxkl=stats[2], ratio=stats[3],
                   nonfinite=self.tail[1].clone(), new_logprobs=new_lp)
        if optimizer_step:
            out["grad_norm"] = self.optimizer_step(grad_scale=1.0 / world, guard=True)
        return out

    def optimizer_step(self, grad_scale: float = 1.0, guard: bool = False) -> torch.Tensor:
        """Fused global-norm clip + AdamW on the flat buffers.  ``guard``: skip the update (on the device, no host sync) when
        the all-reduced non-finite-loss flag of the last ppo_update is set."""
        lib = L.load()
        self.step_count += 1
        with torch.cuda.device(self.device):
            L.check(lib.tpdm_adamw_step(L.ptr(self.params), L.ptr(self.grads), L.ptr(self.m), L.ptr(self.v), self.params.numel(), float(self.lr),
                                        float(self.betas[0]), float(self.betas[1]), float(self.eps), float(self.weight_decay),
                                        float(self.max_grad_norm), self.step_count, float(grad_scale), L.ptr(self.sumsq),
                                        L.ptr(self.conv1_bf16), self.n_conv1, self.tail.data_ptr() + 4 if guard else None, L.stream_ptr()))
        return self.sumsq.sqrt().float()

    # ---- autograd hook for the reference trainer's own loop ----------------------------------------------------------
    def logprobs(self, sigmas: torch.Tensor, tpm_inputs_nhwc: torch.Tensor, tembs: torch.Tensor, min_sigma: float, epsilon: float = 1e-3,
                 relative: bool = True, prediction_type: str = "alpha_beta") -> torch.Tensor:
        """only_predict_logprobs (modeling_sd3_pnt.py:670-726) as a differentiable function of the module's parameters:
        (mb, T) log-probs whose ``.backward()`` deposits into ``time_predictor.<name>.grad`` in PyTorch layouts, so that
        ``accelerator.backward(loss)`` / DDP all-reduce / ``clip_grad_norm_`` / ``optimizer.step`` of the reference trainer
        (rloo_trainer.py:485-523) run unmodified.  Forward and backward are the native kernels."""
        params = [p for _, p in self.module.named_parameters()]
        names = [n for n, _ in self.module.named_parameters()]
        self.load_from_module()      # an external optimizer may have stepped the module since the last call
        return _LogprobReplay.apply(self, names, sigmas, tpm_inputs_nhwc, tembs, float(min_sigma), float(epsilon), bool(relative),
                                    prediction_type, *params)


class _LogprobReplay(torch.autograd.Function):
    """forward: tpdm_tpm_train_forward + tpdm_beta_logprob; backward: dz = dlogprob/dz * grad -> tpdm_tpm_train_backward."""

    @staticmethod
    def forward(ctx, trainer, names, sigmas, x_nhwc, tembs, min_sigma, epsilon, relative, prediction_type, *params):
        lib = L.load()
        mb, T = sigmas.shape
        f32 = dict(device=trainer.device, dtype=torch.float32)
        ab = trainer.forward(x_nhwc.reshape(mb * T, trainer.g, trainer.g, 2 * trainer.D), tembs.reshape(mb * T, trainer.D))
        sig = sigmas.to(**f32).contiguous()
        lp = torch.empty(mb, T, **f32)
        dlp = torch.empty(mb * T, 2, **f32)
        with torch.cuda.device(trainer.device):
            L.check(lib.tpdm_beta_logprob(L.ptr(ab), L.ptr(sig), mb, T, min_sigma, epsilon, 1 if relative else 0,
                                          0 if prediction_type == "alpha_beta" else 1, float(trainer.module.epsilon), L.ptr(lp), L.ptr(dlp),
                                          L.stream_ptr()))
        ctx.trainer, ctx.names, ctx.dlp, ctx.shape, ctx.generation = trainer, names, dlp, (mb, T), trainer._generation
        ctx.param_meta = [(p.shape, p.dtype) for p in params]
        return lp

    @staticmethod
    def backward(ctx, grad_lp):
        trainer = ctx.trainer
        mb, T = ctx.shape
        if trainer._generation != ctx.generation:
            raise RuntimeError("TimePredictor replay: backward() after a later forward() -- the saved activations were overwritten "
                               "(call backward on each micro-batch before replaying the next, as rloo_trainer.py:485-501 does)")
        dz = ctx.dlp * grad_lp.to(device=trainer.device, dtype=torch.float32).reshape(mb * T, 1)
        trainer.backward(dz)
        grads = trainer.tensors(trainer.grads)
        out = [grads[n].to(dt).contiguous() for n, (shape, dt) in zip(ctx.names, ctx.param_meta)]
        return (None,) * 9 + tuple(out)
