"""Host-side engine: packs module weights for libtpdm_b200.so, owns shape-bound plans (workspace + prebuilt TMA
descriptors) and drives the adaptive loop.  PyTorch is used for device memory and streams only; every arithmetic
operation of the path runs inside the C-ABI library (no eager fallback exists).
"""
from __future__ import annotations

import collections
import ctypes as C
import os
import weakref
from typing import Dict, Optional, Tuple

import torch

from . import _lib as L


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(dtype=torch.float32).contiguous()


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(dtype=torch.bfloat16).contiguous()


def _pad_heads_rows(w: torch.Tensor, heads: int, d: int, dp: int) -> torch.Tensor:
    """[heads*d, ...] -> [heads*dp, ...] with zero rows for the padded head dims."""
    if d == dp:
        return w
    rest = w.shape[1:]
    out = w.new_zeros((heads, dp) + tuple(rest))
    out[:, :d] = w.reshape((heads, d) + tuple(rest))
    return out.reshape((heads * dp,) + tuple(rest))


MMDIT_PRECISIONS = ("bf16", "fp8")


def check_mmdit_precision(precision: str) -> str:
    """``"bf16"`` (every MMDiT GEMM in bf16, the default) or ``"fp8"`` (QKV and FF1 of both streams as E4M3 GEMMs)."""
    if precision not in MMDIT_PRECISIONS:
        raise ValueError(f"mmdit_precision must be one of {MMDIT_PRECISIONS}, got {precision!r}")
    return precision


def _fused_rows(g, p: str, names, attn: str, H: int, d: int, dp: int):
    """Fused projection of a block, [len(names) * H * dp, D] weight and bias, each head padded to dp rows (zeros)."""
    w = torch.cat([_pad_heads_rows(g(p + f"{attn}.{n}.weight"), H, d, dp) for n in names], 0)
    bias = torch.cat([_pad_heads_rows(g(p + f"{attn}.{n}.bias"), H, d, dp) for n in names], 0)
    return w, bias


def quantize_fp8_rows(w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """E4M3 codes (uint8, [rows, K]) and fp32 scales ([rows]) of each row of ``w``, by the library kernel
    ``tpdm_quantize_fp8_rows``: w ~= codes.view(torch.float8_e4m3fn).float() * scales[:, None]."""
    lib = L.load()
    x = _f32(w)
    codes = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    scales = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        L.check(lib.tpdm_quantize_fp8_rows(L.ptr(x), x.shape[0], x.shape[1], L.ptr(codes), L.ptr(scales), L.stream_ptr()))
    return codes, scales


class PackedWeights:
    """Device tensors in the layout include/tpdm_b200.h documents, plus the ctypes structs pointing at them."""

    def __init__(self):
        self.keep = []           # owning references
        self.by_name = {}
        self.struct = L.TpdmWeights()
        self.blocks = None
        self.fp8_blocks = None

    def _set(self, struct, name, tensor):
        if struct is self.struct and name in self.by_name:   # refresh: same storage, same pointers (plans stay valid)
            self.by_name[name].copy_(tensor)
            return
        self.keep.append(tensor)
        if struct is self.struct:
            self.by_name[name] = tensor
        setattr(struct, name, tensor.data_ptr())


def pack_transformer(pw: PackedWeights, sd: Dict[str, torch.Tensor], cfg, device) -> None:
    """diffusers-layout state dict of CustomSD3Transformer2DModel -> tpdm_weights (MMDiT part)."""
    H, d = cfg.num_attention_heads, cfg.attention_head_dim
    D = H * d
    dp = 64 if d <= 64 else 128
    Lyr = cfg.num_layers
    dual_layers = set(int(i) for i in (getattr(cfg, "dual_attention_layers", ()) or ()))
    g = lambda k: sd[k].to(device)
    s = pw.struct
    pw._set(s, "patch_w", _f32(g("pos_embed.proj.weight").reshape(D, -1)))
    pw._set(s, "patch_b", _f32(g("pos_embed.proj.bias")))
    pw._set(s, "pos_table", _f32(g("pos_embed.pos_embed").reshape(-1, D)))
    for short, base in (("t", "time_text_embed.timestep_embedder"), ("p", "time_text_embed.text_embedder")):
        pw._set(s, f"{short}_w1", _f32(g(base + ".linear_1.weight")))
        pw._set(s, f"{short}_b1", _f32(g(base + ".linear_1.bias")))
        pw._set(s, f"{short}_w2", _f32(g(base + ".linear_2.weight")))
        pw._set(s, f"{short}_b2", _f32(g(base + ".linear_2.bias")))
    pw._set(s, "ctx_w", _bf16(g("context_embedder.weight")))
    pw._set(s, "ctx_b", _f32(g("context_embedder.bias")))
    pw._set(s, "proj_w", _bf16(g("proj_out.weight")))
    pw._set(s, "proj_b", _f32(g("proj_out.bias")))
    ada_w, ada_b = [], []
    blocks = (L.TpdmBlockWeights * Lyr)()
    for i in range(Lyr):
        p = f"transformer_blocks.{i}."
        last = i == Lyr - 1
        ada_w += [g(p + "norm1.linear.weight"), g(p + "norm1_context.linear.weight")]
        ada_b += [g(p + "norm1.linear.bias"), g(p + "norm1_context.linear.bias")]
        b = blocks[i]

        def fused(names, attn="attn"):
            w, bias = _fused_rows(g, p, names, attn, H, d, dp)
            return _bf16(w), _f32(bias)

        def out_proj(name, attn="attn"):
            w = g(p + f"{attn}.{name}.weight")  # [D, H*d] -> [D, H*dp]
            if d != dp:
                w = _pad_heads_rows(w.t().contiguous(), H, d, dp).t().contiguous()
            return _bf16(w), _f32(g(p + f"{attn}.{name}.bias"))

        for field, (w, bias) in (("qkv", fused(("to_q", "to_k", "to_v"))), ("cqkv", fused(("add_q_proj", "add_k_proj", "add_v_proj"))),
                                 ("out", out_proj("to_out.0"))):
            pw._set(b, field + "_w", w)
            pw._set(b, field + "_b", bias)
        pw._set(b, "ff1_w", _bf16(g(p + "ff.net.0.proj.weight")))
        pw._set(b, "ff1_b", _f32(g(p + "ff.net.0.proj.bias")))
        pw._set(b, "ff2_w", _bf16(g(p + "ff.net.2.weight")))
        pw._set(b, "ff2_b", _f32(g(p + "ff.net.2.bias")))
        if not last:
            w, bias = out_proj("to_add_out")
            pw._set(b, "cout_w", w)
            pw._set(b, "cout_b", bias)
            pw._set(b, "cff1_w", _bf16(g(p + "ff_context.net.0.proj.weight")))
            pw._set(b, "cff1_b", _f32(g(p + "ff_context.net.0.proj.bias")))
            pw._set(b, "cff2_w", _bf16(g(p + "ff_context.net.2.weight")))
            pw._set(b, "cff2_b", _f32(g(p + "ff_context.net.2.bias")))
        dual = i in dual_layers
        if dual:  # SD3.5 attn2 (transformer_sd3.py:138): image-token self-attention with its own projections
            for field, (w, bias) in (("qkv2", fused(("to_q", "to_k", "to_v"), "attn2")), ("out2", out_proj("to_out.0", "attn2"))):
                pw._set(b, field + "_w", w)
                pw._set(b, field + "_b", bias)
        if cfg.qk_norm == "rms_norm":
            names = [("norm_q", "attn.norm_q"), ("norm_k", "attn.norm_k"), ("norm_added_q", "attn.norm_added_q"),
                     ("norm_added_k", "attn.norm_added_k")]
            if dual:
                names += [("norm_q2", "attn2.norm_q"), ("norm_k2", "attn2.norm_k")]
            for field, name in names:
                w = g(p + f"{name}.weight")
                wp = w.new_zeros(dp)
                wp[:d] = w
                pw._set(b, field, _f32(wp))
    ada_w.append(g("norm_out.linear.weight"))
    ada_b.append(g("norm_out.linear.bias"))
    pw._set(s, "adaln_w", _bf16(torch.cat(ada_w, 0)))
    pw._set(s, "adaln_b", _f32(torch.cat(ada_b, 0)))
    assert pw.keep[-1].numel() == 12 * D * Lyr - 2 * D + 3 * D * len(dual_layers)
    pw.blocks = blocks
    s.blocks = C.cast(blocks, C.POINTER(L.TpdmBlockWeights))


def pack_fp8_blocks(pw: PackedWeights, sd: Dict[str, torch.Tensor], cfg, device) -> None:
    """tpdm_fp8_block_weights: E4M3 codes + per-output-channel scales of the fused QKV / context QKV and FF1 / context FF1
    matrices, quantized on the device from the state dict's values."""
    H, d = cfg.num_attention_heads, cfg.attention_head_dim
    dp = 64 if d <= 64 else 128
    Lyr = cfg.num_layers
    g = lambda k: sd[k].to(device)
    blocks = (L.TpdmFp8BlockWeights * Lyr)()
    for i in range(Lyr):
        p = f"transformer_blocks.{i}."
        mats = [("qkv", _fused_rows(g, p, ("to_q", "to_k", "to_v"), "attn", H, d, dp)[0]),
                ("cqkv", _fused_rows(g, p, ("add_q_proj", "add_k_proj", "add_v_proj"), "attn", H, d, dp)[0]),
                ("ff1", g(p + "ff.net.0.proj.weight"))]
        if i != Lyr - 1:
            mats.append(("cff1", g(p + "ff_context.net.0.proj.weight")))
        for field, w in mats:
            codes, scales = quantize_fp8_rows(w)
            pw._set(blocks[i], field + "_w", codes)
            pw._set(blocks[i], field + "_s", scales)
    pw.fp8_blocks = blocks


def pack_time_predictor(pw: PackedWeights, sd: Dict[str, torch.Tensor], device) -> None:
    """TimePredictor state dict (modeling_sd3_pnt.py:85-126 names) -> tpdm_weights (TPM part)."""
    g = lambda k: sd[k].to(device)
    s = pw.struct
    c1 = g("conv1.weight")  # [C1, 2D, 3, 3] -> [C1, 9, 2D]
    pw._set(s, "tpm_conv1_w", _bf16(c1.permute(0, 2, 3, 1).reshape(c1.shape[0], -1)))
    pw._set(s, "tpm_conv1_b", _f32(g("conv1.bias")))
    pw._set(s, "tpm_lin_w", _f32(g("norm1.linear.weight")))
    pw._set(s, "tpm_lin_b", _f32(g("norm1.linear.bias")))
    pw._set(s, "tpm_gn_w", _f32(g("norm1.norm.weight")))
    pw._set(s, "tpm_gn_b", _f32(g("norm1.norm.bias")))
    c2 = g("conv2.weight")  # [oc, c, 3, 3] -> [9, c, oc]
    pw._set(s, "tpm_conv2_w", _f32(c2.permute(2, 3, 1, 0).reshape(9, c2.shape[1], c2.shape[0])))
    pw._set(s, "tpm_conv2_b", _f32(g("conv2.bias")))
    pw._set(s, "tpm_fc1_w", _f32(g("fc1.weight")))
    pw._set(s, "tpm_fc1_b", _f32(g("fc1.bias")))
    pw._set(s, "tpm_fc2_w", _f32(g("fc2.weight")))
    pw._set(s, "tpm_fc2_b", _f32(g("fc2.bias")))


class _FlagReadback:
    """Device int32 flags looked at one step late, so that the device never waits for the host: ``push`` copies them into the
    next row of a pinned ring behind the step just enqueued (one copy, one event record), and a row is looked at once its
    copy has completed.  ``last`` is the newest row looked at (zeros before the first)."""

    def __init__(self, width: int, ring: int = 64):
        self._host = torch.zeros(ring, width, dtype=torch.int32).pin_memory()
        self._events = [torch.cuda.Event() for _ in range(ring)]
        self._pending = collections.deque()      # rows pushed and not looked at, oldest first
        self._pushes = 0
        self.last = [0] * width

    def push(self, src: torch.Tensor) -> None:
        row = self._pushes % len(self._events)
        self._pushes += 1
        self._host[row].copy_(src, non_blocking=True)
        self._events[row].record()
        self._pending.append(row)

    def _take(self) -> list:
        row = self._pending.popleft()
        self._events[row].synchronize()
        self.last = self._host[row].tolist()
        return self.last

    def settle(self) -> Optional[list]:
        """Waits for every push but the newest; returns the newest row that settled (None: none did)."""
        seen = None
        while len(self._pending) > 1:
            seen = self._take()
        return seen

    def poll(self) -> Optional[list]:
        """Looks at the completed rows without blocking; returns the newest (None: none completed since the last look)."""
        seen = None
        while self._pending and self._events[self._pending[0]].query():
            seen = self._take()
        return seen

    def wait_all(self) -> None:
        while self._pending:
            self._take()


class Plan:
    """A shape-bound workspace with typed torch views over the library's state buffers."""

    def __init__(self, engine: "Engine", batch: int, cfg_pairs: bool, latent: int, n_text: int, max_steps: int):
        lib = L.load()
        self.engine, self.batch, self.cfg_pairs, self.latent, self.n_text, self.max_steps = engine, batch, cfg_pairs, latent, n_text, max_steps
        nbytes = lib.tpdm_plan_workspace_bytes(engine.ctx, batch, int(cfg_pairs), latent, latent, n_text, max_steps)
        if nbytes == 0:
            L.check(L.TPDM_ERR_SHAPE if lib.tpdm_last_error() else L.TPDM_ERR_ARG)
        self.workspace, base = L.aligned_workspace(nbytes, engine.device)
        handle = L.vp()
        L.check(lib.tpdm_plan_create(engine.ctx, batch, int(cfg_pairs), latent, latent, n_text, max_steps, base, nbytes, C.byref(handle)))
        self.handle = handle
        self.state = None
        if engine.has_mmdit and engine.has_tpm and cfg_pairs:
            st = L.TpdmSampleState()
            L.check(lib.tpdm_sample_state_get(handle, C.byref(st)))
            cfg, D, g = engine.cfg, engine.D, latent // 2
            Cc = cfg["in_channels"]
            f32, i32 = torch.float32, torch.int32
            view = lambda ptr, dtype, shape: L.view_at(self.workspace, ptr, dtype, shape)
            self.state = dict(
                latents=view(st.latents, f32, (batch, Cc, latent, latent)),
                velocity=view(st.velocity, f32, (batch, Cc, latent, latent)),
                sigma_hist=view(st.sigma_hist, f32, (batch, max_steps + 1)),
                alphas=view(st.alphas, f32, (batch, max_steps)),
                betas=view(st.betas, f32, (batch, max_steps)),
                logprobs=view(st.logprobs, f32, (batch, max_steps)),
                prob_masks=view(st.prob_masks, i32, (batch, max_steps)),
                all_done=view(st.all_done, i32, (max_steps,)),
                tembs=view(st.tembs, f32, (max_steps, batch, D)),
                tpm_input=view(st.tpm_input, torch.bfloat16, (batch, g, g, 2 * D)),
                history_latents=view(st.history_latents, f32, (max_steps, batch, Cc, latent, latent)),
            )

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                L.load().tpdm_plan_destroy(self.handle)
        except Exception:
            pass


class Engine:
    """One per (transformer, time_predictor) pair and device."""

    def __init__(self, cfg: dict, device: torch.device, transformer_sd: Optional[Dict[str, torch.Tensor]] = None, transformer_cfg=None,
                 tpm_sd: Optional[Dict[str, torch.Tensor]] = None, min_sigma: float = 0.001, relative: bool = True,
                 prediction_type: str = "alpha_beta", epsilon: float = 1e-3, tpm_epsilon: float = 1.0, tpm_channels: int = 128,
                 mmdit_precision: str = "bf16"):
        """``mmdit_precision="fp8"`` runs the QKV and FF1 projections of both streams as E4M3 GEMMs (per-token activation
        scales, per-channel weight scales); every other GEMM stays bf16."""
        check_mmdit_precision(mmdit_precision)
        if mmdit_precision == "fp8" and transformer_sd is None:
            raise ValueError("mmdit_precision='fp8' needs the transformer weights")
        lib = L.load()
        if device.type != "cuda":
            raise RuntimeError("tpdm_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        if prediction_type not in ("alpha_beta", "mode_concentration"):
            raise ValueError(f"unknown prediction_type {prediction_type!r}")
        self.cfg, self.device, self.mmdit_precision = dict(cfg), device, mmdit_precision
        self.D = cfg["num_attention_heads"] * cfg["attention_head_dim"]
        c = L.TpdmConfig(
            num_layers=cfg["num_layers"], num_heads=cfg["num_attention_heads"], head_dim=cfg["attention_head_dim"],
            joint_attention_dim=cfg["joint_attention_dim"], pooled_projection_dim=cfg["pooled_projection_dim"],
            in_channels=cfg["in_channels"], out_channels=cfg["out_channels"], patch_size=cfg["patch_size"],
            pos_embed_max_size=cfg["pos_embed_max_size"], qk_norm=1 if cfg.get("qk_norm") == "rms_norm" else 0,
            tpm_channels=tpm_channels, prediction_type=0 if prediction_type == "alpha_beta" else 1, relative=1 if relative else 0,
            min_sigma=min_sigma, epsilon=epsilon, tpm_epsilon=tpm_epsilon,
            dual_attention_mask=sum(1 << int(i) for i in set(cfg.get("dual_attention_layers", ()) or ())))
        with torch.cuda.device(device):
            handle = L.vp()
            L.check(lib.tpdm_create(C.byref(c), C.byref(handle)))
            self.ctx = handle
            self.weights = PackedWeights()
            self.has_mmdit = transformer_sd is not None
            self.has_tpm = tpm_sd is not None
            if self.has_mmdit:
                pack_transformer(self.weights, transformer_sd, transformer_cfg, device)
            if self.has_tpm:
                pack_time_predictor(self.weights, tpm_sd, device)
            L.check(lib.tpdm_set_weights(self.ctx, C.byref(self.weights.struct)))
            if mmdit_precision == "fp8":
                pack_fp8_blocks(self.weights, transformer_sd, transformer_cfg, device)
                L.check(lib.tpdm_set_fp8_weights(self.ctx, self.weights.fp8_blocks))
        self.plans: Dict[Tuple, Plan] = {}
        self._streams = weakref.WeakSet()    # open PromptStreams: they read the packed weights from their own CUDA stream
        self._sample_flags, self._queue_flags = _FlagReadback(1), _FlagReadback(1)    # all_done[step] / active slots
        self.min_sigma = min_sigma

    def __del__(self):
        try:
            self.plans.clear()
            if getattr(self, "ctx", None):
                L.load().tpdm_destroy(self.ctx)
        except Exception:
            pass

    def refresh_time_predictor(self, tpm_sd: Dict[str, torch.Tensor]) -> None:
        """Copy new TimePredictor values into the already packed device tensors (pointers and TMA descriptors unchanged)."""
        if not self.has_tpm:
            raise RuntimeError("engine was built without a TimePredictor")
        busy = [st for st in self._streams if st._open and st._harvested != st._submitted]
        if busy:
            raise RuntimeError("the TimePredictor weights cannot change while an open prompt stream has requests in flight: their "
                               "trajectories would switch weights part-way (drain or close the stream first)")
        cur = torch.cuda.current_stream(self.device)
        for st in self._streams:            # the copies run after the stream's queued steps and before its next ones
            if st._open:
                cur.wait_stream(st._cs)
        with torch.cuda.device(self.device):
            pack_time_predictor(self.weights, tpm_sd, self.device)
        for st in self._streams:
            if st._open:
                st._cs.wait_stream(cur)

    def plan(self, batch: int, cfg_pairs: bool, latent: int, n_text: int, max_steps: int = 1) -> Plan:
        key = (batch, bool(cfg_pairs), latent, n_text, max_steps)
        p = self.plans.get(key)
        if p is None:
            if len(self.plans) >= 4:  # bound the HBM held by cached workspaces
                self.plans.pop(next(iter(self.plans)))
            with torch.cuda.device(self.device):
                p = Plan(self, batch, cfg_pairs, latent, n_text, max_steps)
            self.plans[key] = p
        return p

    # ---- CustomSD3Transformer2DModel.forward -------------------------------------------------------------------
    def mmdit_forward(self, hidden_states, encoder_hidden_states, pooled_projections, timestep):
        lib = L.load()
        Bt, Cc, h, w = hidden_states.shape
        if h != w:
            raise ValueError(f"only square latents are supported (got {h}x{w})")
        n_text = encoder_hidden_states.shape[1]
        plan = self.plan(Bt, False, h, n_text, 1)
        dev, f32 = self.device, torch.float32
        lat = hidden_states.to(device=dev, dtype=f32).contiguous()
        enc = encoder_hidden_states.to(device=dev, dtype=f32).contiguous()
        pooled = pooled_projections.to(device=dev, dtype=f32).contiguous()
        ts = timestep.to(device=dev, dtype=f32).reshape(-1)
        if ts.numel() == 1:
            ts = ts.expand(Bt)
        ts = ts.contiguous()
        if enc.shape[0] != Bt or pooled.shape[0] != Bt or ts.shape[0] != Bt:
            raise ValueError("batch sizes of hidden_states / encoder_hidden_states / pooled_projections / timestep differ")
        N = (h // 2) * (w // 2)
        out = torch.empty(Bt, self.cfg["out_channels"], h, w, device=dev, dtype=f32)
        temb = torch.empty(Bt, self.D, device=dev, dtype=f32)
        h1 = torch.empty(Bt, N, self.D, device=dev, dtype=f32)
        h2 = torch.empty(Bt, N, self.D, device=dev, dtype=f32)
        with torch.cuda.device(dev):
            L.check(lib.tpdm_mmdit_forward(plan.handle, L.ptr(lat), L.ptr(ts), L.ptr(enc), L.ptr(pooled), L.ptr(out), L.ptr(temb),
                                           L.ptr(h1), L.ptr(h2), L.stream_ptr()))
        return out, temb, h1, h2

    # ---- TimePredictor.forward ---------------------------------------------------------------------------------
    def tpm_forward(self, x, temb):
        lib = L.load()
        B, C2, g, g2 = x.shape
        if g != g2 or C2 != 2 * self.D:
            raise ValueError(f"TimePredictor input must be (B, {2 * self.D}, g, g); got {tuple(x.shape)}")
        plan = self.plan(B, False, 2 * g, 8, 1)
        dev, f32 = self.device, torch.float32
        xx = x.to(device=dev, dtype=f32).contiguous()
        tt = temb.to(device=dev, dtype=f32).contiguous()
        out = torch.empty(B, 2, device=dev, dtype=f32)
        with torch.cuda.device(dev):
            L.check(lib.tpdm_tpm_forward(plan.handle, L.ptr(xx), L.ptr(tt), L.ptr(out), L.stream_ptr()))
        return out

    # ---- the adaptive loop -------------------------------------------------------------------------------------
    def sample(self, latents, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds,
               max_inference_steps: int, guidance_scale: float, predict: bool, ratios=None, seed: int = 0,
               record_tpm_inputs: bool = False, record_velocity: bool = False, use_graph: Optional[bool] = None):
        """Runs tpdm_sample_step until every sigma_next < min_sigma (checked one step late through a pinned flag, the
        speculative extra step is skipped on the device) or max_inference_steps.  Returns a dict of device tensors.
        ``use_graph`` (default: on, ``TPDM_SAMPLE_GRAPH=0`` turns it off): every step index is replayed from a CUDA graph
        captured the first time it runs on the plan (~190 launches become one ``cudaGraphLaunch``); the trajectory then runs on a
        side stream, because the legacy default stream cannot be captured, and the caller's stream waits for it."""
        lib = L.load()
        if use_graph is None:
            use_graph = os.environ.get("TPDM_SAMPLE_GRAPH", "1") != "0"
        B, Cc, h, w = latents.shape
        dev, f32 = self.device, torch.float32
        plan = self.plan(B, True, h, prompt_embeds.shape[1], max_inference_steps)
        st = plan.state
        cvt = lambda t: t.to(device=dev, dtype=f32).contiguous()
        lat, pe, ne, pp, npp = cvt(latents), cvt(prompt_embeds), cvt(negative_prompt_embeds), cvt(pooled_prompt_embeds), cvt(negative_pooled_prompt_embeds)
        rt = None
        if not predict and ratios is not None:
            rt = cvt(ratios)
            if rt.shape != (B, max_inference_steps):
                raise ValueError(f"ratios must have shape {(B, max_inference_steps)}")
        rec = vel = None
        g = h // 2
        if record_tpm_inputs:
            rec = torch.empty(B, max_inference_steps, g, g, 2 * self.D, device=dev, dtype=torch.bfloat16)
        if record_velocity:
            vel = torch.empty(B, max_inference_steps, Cc, h, w, device=dev, dtype=f32)
        flags = self._sample_flags
        executed = max_inference_steps
        step_fn = lib.tpdm_sample_step_graph if use_graph else lib.tpdm_sample_step
        side = None
        if use_graph:
            side = getattr(self, "_sample_stream", None)
            if side is None:
                side = self._sample_stream = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev), torch.cuda.stream(side):
            stream = L.stream_ptr()
            L.check(lib.tpdm_sample_begin(plan.handle, L.ptr(lat), L.ptr(ne), L.ptr(pe), L.ptr(npp), L.ptr(pp), float(guidance_scale),
                                          1 if predict else 0, L.ptr(rt) if rt is not None else None, int(seed) & (2**64 - 1), stream))
            for step in range(max_inference_steps):
                L.check(step_fn(plan.handle, step, stream))
                if rec is not None:
                    rec[:, step].copy_(st["tpm_input"])
                if vel is not None:
                    vel[:, step].copy_(st["velocity"])
                flags.push(st["all_done"][step: step + 1])
                done = flags.settle()      # the flag of the previous step: the device never waits for the host
                if step >= 1 and done[0] != 0:
                    executed = step  # steps [0, step) are real; step `step` was skipped on the device
                    break
            else:
                flags.wait_all()
        if side is not None:
            torch.cuda.current_stream(dev).wait_stream(side)
            for t in (lat, pe, ne, pp, npp, rt, rec, vel):
                if t is not None:
                    t.record_stream(side)
        T = executed
        out = dict(
            steps=T,
            sigmas=st["sigma_hist"][:, 1: T + 1].clone(), alphas=st["alphas"][:, :T].clone(), betas=st["betas"][:, :T].clone(),
            logprobs_raw=st["logprobs"][:, :T].clone(), prob_masks=st["prob_masks"][:, :T].clone().bool(),
            tembs=st["tembs"][:T].permute(1, 0, 2).clone(), history_latents=st["history_latents"][:T].permute(1, 0, 2, 3, 4).clone(),
        )
        if rec is not None:
            out["tpm_inputs_nhwc"] = rec[:, :T]
        if vel is not None:
            out["velocities"] = vel[:, :T]
        return out

    def _probe_and_order(self, lat, pe, ne, pp, npp, guidance_scale, max_steps, out_lat, out_steps, out_sig):
        """Longest-expected-first scheduling for the device queue.  Greedy list scheduling loses the tail: the last GPUs to finish
        are whoever drew a long prompt late (86.6 % of the sum-of-steps / N bound on 8 GPUs, profiles/r01_config3_devq_n8.log).
        Trajectory lengths are not known in advance, but the FIRST TimePredictor call already says how fast sigma falls for a
        prompt.  So every GPU runs denoising step 0 for its static share of the prompts (one batched call; the step is not wasted:
        it IS step 0 of those trajectories), the post-step latents and sigmas are all-gathered (1 MB per prompt over NVLink -- the
        one exchange of this scheduler, a few hundred microseconds), every rank sorts the prompts by the expected number of
        remaining steps, ceil(log(min_sigma / sigma_1) / log(sigma_1)), and the queue hands them out longest first with every
        prompt entering at step 1.  Ticket claiming stays dynamic, so a wrong estimate costs balance, never correctness: each
        prompt still follows exactly its own trajectory.  Returns (latents after step 0 [P], order, n_queued, sigma_1 [P])."""
        import torch.distributed as dist

        lib = L.load()
        P = lat.shape[0]
        dev = self.device
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        rank = dist.get_rank() if world > 1 else 0
        if P % world != 0:
            raise ValueError(f"schedule='lpt' needs the number of prompts ({P}) to be a multiple of the number of ranks ({world})")
        mine = torch.arange(rank, P, world, device=dev)
        nb = mine.numel()
        plan = self.plan(nb, True, lat.shape[-1], pe.shape[1], 1)
        st = plan.state
        sel = lambda t: t[mine].contiguous()
        l0, pe0, ne0, pp0, npp0 = sel(lat), sel(pe), sel(ne), sel(pp), sel(npp)
        with torch.cuda.device(dev):
            stream = L.stream_ptr()
            L.check(lib.tpdm_sample_begin(plan.handle, L.ptr(l0), L.ptr(ne0), L.ptr(pe0), L.ptr(npp0), L.ptr(pp0), float(guidance_scale), 1, None,
                                          0, stream))
            L.check(lib.tpdm_sample_step(plan.handle, 0, stream))
        packed = torch.cat([st["latents"].reshape(nb, -1), st["sigma_hist"][:, 1:2]], dim=1).contiguous()     # (nb, C*h*w + 1)
        if world > 1:
            allp = torch.empty(world, nb, packed.shape[1], device=dev, dtype=packed.dtype)
            dist.all_gather_into_tensor(allp, packed)
            allp = allp.permute(1, 0, 2).reshape(P, -1)          # prompt p = rank + k * world  ->  row k * world + rank = p
        else:
            allp = packed
        lat1 = allp[:, :-1].reshape(lat.shape).contiguous()
        sig1 = allp[:, -1].contiguous()
        from .work_queue import expected_remaining_steps, longest_first_order

        done = sig1 < self.min_sigma                              # the whole trajectory was one step (:608)
        order = longest_first_order(expected_remaining_steps(sig1, self.min_sigma, max_steps)).contiguous()
        n_queued = int((~done).sum().item())
        out_sig[:, 0] = 1.0
        out_sig[:, 1] = sig1
        probed_here = torch.zeros(P, dtype=torch.bool, device=dev)
        probed_here[mine] = True
        fin = done & probed_here                                  # finished at the probe: reported by the rank that ran it
        out_steps[fin] = 1
        out_lat[fin] = lat1[fin]
        return lat1, order, n_queued, sig1

    def sample_queue(self, latents, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds,
                     slots: int, max_inference_steps: int, guidance_scale: float, ticket: Optional[torch.Tensor] = None,
                     out_latents: Optional[torch.Tensor] = None, use_graph: bool = True, schedule: str = "fifo", predict: bool = True,
                     seed: int = 0, ratios: Optional[torch.Tensor] = None, record: bool = True):
        """Device-side prompt queue (``tpdm_queue_*``): all P prompts are resident, ``slots`` of them are in flight; a slot
        whose trajectory ends takes the next ticket on the device.  ``ticket`` (int32 device tensor of one element, zeroed by
        its owner) may be shared between GPUs, which then split one prompt list between them.  Returns device tensors:
        latents (P, C, h, w), steps (P,) (0 for prompts another GPU processed), sigmas (P, max_steps + 1).
        ``predict=False`` samples rollouts (``tpdm_queue_set_rollout``): prompt p follows row p of one lockstep
        ``sample(..., predict=False)`` of all P prompts -- the injected ``ratios`` (P, max_steps) or the device draws of ``seed``.
        The result then also holds alphas, betas, logprobs_raw (P, max_steps), tembs (P, max_steps, D) and, with ``record``,
        tpm_inputs_nhwc (P, max_steps, g, g, 2D) bf16.  They are zero past each prompt's last step: the PPO replay runs the
        TimePredictor on every (prompt, step) and multiplies those inputs by a zero gradient, which a stray NaN would poison."""
        lib = L.load()
        P, Cc, h, w = latents.shape
        dev, f32 = self.device, torch.float32
        if schedule not in ("fifo", "lpt"):
            raise ValueError(f"unknown queue schedule {schedule!r} ('fifo': tickets in prompt order, 'lpt': longest expected trajectory first)")
        if schedule == "lpt" and not predict:
            raise ValueError("schedule='lpt' probes step 0 with the Beta mode and cannot start sampled rollouts (predict=False)")
        if not 1 <= slots <= P:
            raise ValueError(f"slots must be in [1, {P}]")
        cvt = lambda t: t.to(device=dev, dtype=f32).contiguous()
        lat, pe, ne, pp, npp = cvt(latents), cvt(prompt_embeds), cvt(negative_prompt_embeds), cvt(pooled_prompt_embeds), cvt(negative_pooled_prompt_embeds)
        rt, rec = None, {}
        if not predict:
            if ratios is not None:
                rt = cvt(ratios)
                if rt.shape != (P, max_inference_steps):
                    raise ValueError(f"ratios must have shape {(P, max_inference_steps)}, got {tuple(rt.shape)}")
            z = lambda *s, dtype=f32: torch.zeros(*s, device=dev, dtype=dtype)
            rec = dict(alphas=z(P, max_inference_steps), betas=z(P, max_inference_steps), logprobs_raw=z(P, max_inference_steps))
            rec["tembs"] = z(P, max_inference_steps, self.D)
            if record:
                g = h // 2
                rec["tpm_inputs_nhwc"] = z(P, max_inference_steps, g, g, 2 * self.D, dtype=torch.bfloat16)
        if ticket is None:
            ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        out_lat = torch.zeros(P, Cc, h, w, device=dev, dtype=f32) if out_latents is None else out_latents
        out_steps = torch.zeros(P, dtype=torch.int32, device=dev)
        out_sig = torch.zeros(P, max_inference_steps + 1, device=dev, dtype=f32)
        order = init_sigma = None
        n_queued, init_step = P, 0
        if schedule == "lpt" and max_inference_steps > 1:
            lat, order, n_queued, init_sigma = self._probe_and_order(lat, pe, ne, pp, npp, guidance_scale, max_inference_steps, out_lat, out_steps, out_sig)
            init_step = 1
            if n_queued == 0:       # every trajectory ended at its first step
                return dict(latents=out_lat, steps=out_steps, sigmas=out_sig, device_steps=1)
        plan = self.plan(slots, True, h, prompt_embeds.shape[1], max_inference_steps)
        nbytes = lib.tpdm_queue_workspace_bytes(plan.handle, P)
        ws, base = L.aligned_workspace(nbytes, dev)
        flags = self._queue_flags
        # the step is replayed from a CUDA graph (captured on the first step), which needs a non-default stream
        qs = getattr(self, "_queue_stream", None)
        if qs is None:
            qs = self._queue_stream = torch.cuda.Stream(device=dev)
        qs.wait_stream(torch.cuda.current_stream(dev))
        step_fn = lib.tpdm_queue_step_graph if use_graph else lib.tpdm_queue_step
        with torch.cuda.device(dev), torch.cuda.stream(qs):
            stream = L.stream_ptr()
            L.check(lib.tpdm_queue_begin(plan.handle, P, L.ptr(lat), L.ptr(ne), L.ptr(pe), L.ptr(npp), L.ptr(pp), float(guidance_scale), base,
                                         nbytes, ticket.data_ptr(), L.ptr(out_lat), L.ptr(out_steps), L.ptr(out_sig),
                                         L.ptr(order) if order is not None else None, int(n_queued),
                                         L.ptr(init_sigma) if init_sigma is not None else None, int(init_step), stream))
            if not predict:
                L.check(lib.tpdm_queue_set_rollout(plan.handle, int(seed) & (2**64 - 1), L.ptr(rt), L.ptr(rec["alphas"]), L.ptr(rec["betas"]),
                                                   L.ptr(rec["logprobs_raw"]), L.ptr(rec.get("tembs")), L.ptr(rec.get("tpm_inputs_nhwc"))))
            act_p, slot_p = L.vp(), L.vp()
            L.check(lib.tpdm_queue_status(plan.handle, C.byref(act_p), C.byref(slot_p)))
            active = L.view_at(ws, act_p.value, torch.int32, (1,))     # the counters live in the queue workspace
            limit = (P + slots - 1) // slots * max_inference_steps + 2 * max_inference_steps   # upper bound on device steps
            steps_run = 0
            drained = False
            for it in range(limit):
                L.check(step_fn(plan.handle, stream))
                steps_run += 1
                flags.push(active)
                prev = flags.settle()      # the count after the previous step: the device never waits for the host
                if it >= 1 and prev[0] == 0:
                    drained = True
                    break
            if not drained:
                torch.cuda.current_stream().synchronize()
                if int(active.item()) != 0:
                    raise RuntimeError("sample_queue: the queue did not drain within the step bound")
            torch.cuda.current_stream().synchronize()
            flags.wait_all()
        torch.cuda.current_stream(dev).wait_stream(qs)
        self._queue_keepalive = (ws, lat, pe, ne, pp, npp, ticket, order, init_sigma, rt)
        return dict(latents=out_lat, steps=out_steps, sigmas=out_sig, device_steps=steps_run + (1 if init_step else 0), **rec)

    def open_stream(self, slots: int, capacity: int, max_inference_steps: int, guidance_scale: float, use_graph: bool = True, *,
                    latent: int, n_text: int = 333, prepare_latents=None) -> "PromptStream":
        """An open device-side prompt queue (``tpdm_stream_*``): ``slots`` prompts in flight, up to ``capacity`` admitted and not
        yet collected, prompts submitted while it runs.  The stream owns a private plan (outside ``self.plans``) and CUDA stream,
        so ``sample``, ``sample_queue`` and ``mmdit_forward`` calls on this engine stay independent of it.  ``latent`` is the
        latent side, ``n_text`` the text length every prompt must have; ``prepare_latents(n, generator, dtype)`` draws latents for
        a ``submit`` without them."""
        return PromptStream(self, slots, capacity, max_inference_steps, guidance_scale, use_graph, latent, n_text, prepare_latents)


class PromptStream:
    """Continuous batching for serving: ``submit`` admits prompts into the running queue, ``step`` runs denoising steps (every slot
    whose trajectory ends takes the next submitted prompt on the device), ``results`` returns the requests that finished.  Each
    request gets what batch-1 ``forward(predict=True)`` gives it.  Everything runs on the stream's own CUDA stream; the host
    looks at the device counters one step late, so it never stalls the device while prompts are in flight.  The stream reads the
    engine's packed weights: a TimePredictor refresh (``Engine.refresh_time_predictor``, which ``get_engine`` makes after an
    optimizer step) raises RuntimeError while requests are in flight, and is ordered against the stream's steps otherwise."""

    def __init__(self, engine: Engine, slots: int, capacity: int, max_steps: int, guidance_scale: float, use_graph: bool, latent: int,
                 n_text: int, prepare_latents=None):
        if slots < 1 or capacity < 1:
            raise ValueError(f"slots ({slots}) and capacity ({capacity}) must be positive")
        if not (engine.has_mmdit and engine.has_tpm):
            raise RuntimeError("a prompt stream needs both MMDiT and TimePredictor weights")
        lib = L.load()
        dev = engine.device
        self.engine, self.slots, self.capacity, self.max_steps, self.latent, self.n_text = engine, slots, capacity, max_steps, latent, n_text
        self._prepare_latents = prepare_latents
        self._step_fn = lib.tpdm_queue_step_graph if use_graph else lib.tpdm_queue_step
        with torch.cuda.device(dev):
            self._plan = Plan(engine, slots, True, latent, n_text, max_steps)    # private: never handed out by Engine.plan
            self._cs = torch.cuda.Stream(device=dev)
            nbytes = lib.tpdm_stream_workspace_bytes(self._plan.handle, capacity)
            self._ws, base = L.aligned_workspace(nbytes, dev)
            self._cs.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(self._cs):
                L.check(lib.tpdm_stream_open(self._plan.handle, capacity, float(guidance_scale), base, nbytes, L.stream_ptr()))
            self._open = True
            engine._streams.add(self)
            ptrs = [L.vp() for _ in range(5)]
            L.check(lib.tpdm_stream_status(self._plan.handle, *[C.byref(p) for p in ptrs]))
        Cc = engine.cfg["in_channels"]
        view = lambda p, dtype, shape: L.view_at(self._ws, p.value, dtype, shape)
        self._counters = view(ptrs[0], torch.int32, (6,))            # submitted, claimed, completed, executed, active, skip flag
        self._log = view(ptrs[1], torch.int32, (capacity,))
        self._out_lat = view(ptrs[2], torch.float32, (capacity, Cc, latent, latent))
        self._out_steps = view(ptrs[3], torch.int32, (capacity,))
        self._out_sig = view(ptrs[4], torch.float32, (capacity, max_steps + 1))
        self._flags = _FlagReadback(6)
        self._free = list(range(capacity - 1, -1, -1))
        self._entry_req = {}                     # entry -> request id
        self._next_id = self._submitted = self._harvested = 0
        self._freed = []                         # events after the copies out of entries freed since the last submit

    def _check_open(self):
        if not self._open:
            raise RuntimeError("the prompt stream is closed")

    # ---- admission ---------------------------------------------------------------------------------------------
    def submit(self, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds, latents=None,
               generator=None) -> list:
        """Admit n prompts; returns their request ids (increasing).  Latents default to ``prepare_latents`` (as ``forward`` draws
        them).  A ring without n free entries raises RuntimeError and admits nothing."""
        self._check_open()
        eng, dev, f32 = self.engine, self.engine.device, torch.float32
        n = prompt_embeds.shape[0]
        J, PD, Cc = eng.cfg["joint_attention_dim"], eng.cfg["pooled_projection_dim"], eng.cfg["in_channels"]
        if latents is None:
            if self._prepare_latents is None:
                raise ValueError("latents are required (this stream has no latent sampler)")
            latents = self._prepare_latents(n, generator, prompt_embeds.dtype)
        want = dict(prompt_embeds=(n, self.n_text, J), negative_prompt_embeds=(n, self.n_text, J), pooled_prompt_embeds=(n, PD),
                    negative_pooled_prompt_embeds=(n, PD), latents=(n, Cc, self.latent, self.latent))
        got = dict(prompt_embeds=prompt_embeds, negative_prompt_embeds=negative_prompt_embeds, pooled_prompt_embeds=pooled_prompt_embeds,
                   negative_pooled_prompt_embeds=negative_pooled_prompt_embeds, latents=latents)
        for k, shape in want.items():
            if tuple(got[k].shape) != shape:
                raise ValueError(f"{k} must have shape {shape} (text length {self.n_text}), got {tuple(got[k].shape)}")
        if n < 1:
            raise ValueError("submit needs at least one prompt")
        if n > len(self._free):
            raise RuntimeError(f"the prompt stream is full: {n} prompts for {len(self._free)} free entries of {self.capacity}")
        cvt = lambda t: t.to(device=dev, dtype=f32).contiguous()
        ts = [cvt(latents), cvt(negative_prompt_embeds), cvt(prompt_embeds), cvt(negative_pooled_prompt_embeds), cvt(pooled_prompt_embeds)]
        entries = self._free[len(self._free) - n:][::-1]       # taken off the free list only once the library accepted them
        ids = (C.c_int * n)(*entries)
        self._cs.wait_stream(torch.cuda.current_stream(dev))   # the inputs
        for ev in self._freed:
            self._cs.wait_event(ev)
        with torch.cuda.device(dev), torch.cuda.stream(self._cs):
            L.check(L.load().tpdm_stream_submit(self._plan.handle, n, ids, *[L.ptr(t) for t in ts], L.stream_ptr()))
        del self._free[len(self._free) - n:]
        self._freed.clear()
        for t in ts:
            t.record_stream(self._cs)            # alive until the admission kernels have read them
        rids = list(range(self._next_id, self._next_id + n))
        self._entry_req.update(zip(entries, rids))
        self._next_id += n
        self._submitted += n
        return rids

    # ---- steps -------------------------------------------------------------------------------------------------
    def _idle(self) -> bool:
        # no slot held a prompt after the newest step looked at, and nothing was submitted since
        last = self._flags.last
        return last[4] == 0 and last[0] == self._submitted

    def step(self, n: int = 1) -> None:
        """Enqueue up to n denoising steps.  Stops (launching nothing) once no slot is active and nothing is pending."""
        self._check_open()
        dev = self.engine.device
        with torch.cuda.device(dev), torch.cuda.stream(self._cs):
            stream = L.stream_ptr()
            for _ in range(n):
                self._flags.poll()
                if self._idle():
                    break
                L.check(self._step_fn(self._plan.handle, stream))
                self._flags.push(self._counters)
                self._flags.settle()           # the flags of the previous step: the device never waits for the host

    @property
    def device_steps(self) -> int:
        """Denoising steps the device executed (steps skipped on an idle stream are not counted)."""
        self._check_open()
        self._flags.wait_all()
        return int(self._flags.last[3])

    # ---- completions -------------------------------------------------------------------------------------------
    def results(self) -> dict:
        """``{request id: dict(latents (C, h, w), steps, sigmas (steps,))}`` of the requests finished since the last call, as far as
        the host has seen (one step late); their entries are free again."""
        self._check_open()
        self._flags.poll()
        done = self._flags.last[2]
        if done == self._harvested:
            return {}
        dev = self.engine.device
        cur = torch.cuda.current_stream(dev)
        with torch.cuda.device(dev):
            # those log entries and outputs were written by steps that have completed; the steps queued after them do not touch them
            k = torch.arange(self._harvested, done, device=dev) % self.capacity
            ents = self._log[k].long()
            steps = self._out_steps[ents].tolist()
            lat = self._out_lat[ents].clone()
            sig = self._out_sig[ents].clone()
        out = {}
        for j, (e, s) in enumerate(zip(ents.tolist(), steps)):
            out[self._entry_req.pop(e)] = dict(latents=lat[j], steps=s, sigmas=sig[j, 1: s + 1])
            self._free.append(e)
        self._harvested = done
        ev = torch.cuda.Event()
        ev.record(cur)                         # the next admission, which may reuse these entries, runs after these copies
        self._freed.append(ev)
        return out

    def drain(self) -> dict:
        """Step until every submitted request has finished; returns the results not collected yet."""
        self._check_open()
        out = {}
        bound = (self._submitted - self._harvested + self.slots - 1) // self.slots * self.max_steps + 2 * self.max_steps + 4
        for _ in range(bound):
            out.update(self.results())
            if self._harvested == self._submitted:
                return out
            self.step()
            if self._idle():
                self._flags.wait_all()
        out.update(self.results())
        if self._harvested != self._submitted:
            raise RuntimeError("the prompt stream did not drain within the step bound")
        return out

    def close(self) -> None:
        if not self._open:
            return
        self._cs.synchronize()
        L.check(L.load().tpdm_stream_close(self._plan.handle))
        self._open = False
        self.engine._streams.discard(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
