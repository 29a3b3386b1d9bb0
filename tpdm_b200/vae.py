"""VAE decode of the final latent on the native path (SURVEY.md section 8(f) rank 1).

Mirrors the part of diffusers' ``AutoencoderKL`` that the reference touches
(/root/reference/src/models/stable_diffusion_3/modeling_sd3_pnt.py:144-146 construction, :181-184 ``config.block_out_channels``,
:631 / :653-655 ``config.scaling_factor`` / ``config.shift_factor`` / ``decode(z, return_dict=False)[0]``): same class
name, ``.config`` attributes, ``.decode`` signature and state-dict names (``decoder.up_blocks.1.resnets.0.conv1.weight`` ...),
so ``vae.load_state_dict(load_file("vae/diffusion_pytorch_model.safetensors"), strict=False)`` works.  The torch modules
below only HOLD parameters; every FLOP of ``decode`` runs in ``libtpdm_b200.so`` (``tpdm_vae_decode``, csrc/vae.cu).  There
is no encoder and no CPU path."""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib as L


class _Resnet(nn.Module):
    def __init__(self, cin: int, cout: int, groups: int):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=1e-6)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.norm2 = nn.GroupNorm(groups, cout, eps=1e-6)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        if cin != cout:
            self.conv_shortcut = nn.Conv2d(cin, cout, 1)


class _Attention(nn.Module):
    def __init__(self, channels: int, groups: int):
        super().__init__()
        self.group_norm = nn.GroupNorm(groups, channels, eps=1e-6)
        self.to_q, self.to_k, self.to_v = nn.Linear(channels, channels), nn.Linear(channels, channels), nn.Linear(channels, channels)
        self.to_out = nn.ModuleList([nn.Linear(channels, channels), nn.Identity()])


class _MidBlock(nn.Module):
    def __init__(self, channels: int, groups: int):
        super().__init__()
        self.resnets = nn.ModuleList([_Resnet(channels, channels, groups), _Resnet(channels, channels, groups)])
        self.attentions = nn.ModuleList([_Attention(channels, groups)])


class _Upsampler(nn.Module):
    def __init__(self, channels: int):
        super().__init__()
        self.conv = nn.Conv2d(channels, channels, 3, padding=1)


class _UpBlock(nn.Module):
    def __init__(self, cin: int, cout: int, layers: int, groups: int, upsample: bool):
        super().__init__()
        self.resnets = nn.ModuleList([_Resnet(cin if i == 0 else cout, cout, groups) for i in range(layers)])
        if upsample:
            self.upsamplers = nn.ModuleList([_Upsampler(cout)])


class _Decoder(nn.Module):
    def __init__(self, latent_channels, out_channels, block_out_channels, layers_per_block, groups):
        super().__init__()
        ch = list(reversed(block_out_channels))
        self.conv_in = nn.Conv2d(latent_channels, ch[0], 3, padding=1)
        self.mid_block = _MidBlock(ch[0], groups)
        blocks, prev = [], ch[0]
        for i, c in enumerate(ch):
            blocks.append(_UpBlock(prev, c, layers_per_block + 1, groups, i != len(ch) - 1))
            prev = c
        self.up_blocks = nn.ModuleList(blocks)
        self.conv_norm_out = nn.GroupNorm(groups, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], out_channels, 3, padding=1)


def _conv_w(conv: nn.Conv2d, dev, pad_in: int = 0, pad_out: int = 0) -> torch.Tensor:
    """(Cout, Cin, 3, 3) -> bf16 [Cout(+pad)][9][Cin(+pad)] (tap-major), the K layout of the implicit-GEMM convolution"""
    w = conv.weight.detach().to(dev, torch.float32).permute(0, 2, 3, 1)          # Cout, ky, kx, Cin
    co, _, _, ci = w.shape
    out = torch.zeros(max(co, pad_out), 3, 3, max(ci, pad_in), device=dev)
    out[:co, :, :, :ci] = w
    return out.reshape(out.shape[0], -1).to(torch.bfloat16).contiguous()


def _f32(t: torch.Tensor, dev, pad: int = 0) -> torch.Tensor:
    v = t.detach().to(dev, torch.float32).reshape(-1)
    if pad > v.numel():
        v = torch.cat([v, torch.zeros(pad - v.numel(), device=dev)])
    return v.contiguous()


class AutoencoderKL(nn.Module):
    """Decode-only AutoencoderKL (SD3 configuration: no quant / post-quant convolutions)."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3, latent_channels: int = 16,
                 block_out_channels: Sequence[int] = (128, 256, 512, 512), layers_per_block: int = 2, norm_num_groups: int = 32,
                 scaling_factor: float = 1.5305, shift_factor: float = 0.0609, device=None, dtype=None):
        super().__init__()
        self.config = SimpleNamespace(in_channels=in_channels, out_channels=out_channels, latent_channels=latent_channels,
                                      block_out_channels=tuple(block_out_channels), layers_per_block=layers_per_block,
                                      norm_num_groups=norm_num_groups, scaling_factor=scaling_factor, shift_factor=shift_factor,
                                      use_quant_conv=False, use_post_quant_conv=False, mid_block_add_attention=True)
        self.decoder = _Decoder(latent_channels, out_channels, tuple(block_out_channels), layers_per_block, norm_num_groups)
        if device is not None or dtype is not None:
            self.to(device=device, dtype=dtype)
        self.requires_grad_(False).eval()
        self._ctx = None
        self._packed: Optional[List] = None
        self._workspace = None

    # ---- the reference reads these -------------------------------------------------------------------------------
    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    # ---- native context --------------------------------------------------------------------------------------------
    def _ensure_ctx(self):
        if self._ctx is not None:
            return
        lib = L.load()
        c = self.config
        cfg = L.TpdmVaeConfig(latent_channels=c.latent_channels, out_channels=c.out_channels, num_levels=len(c.block_out_channels),
                              layers_per_block=c.layers_per_block, norm_num_groups=c.norm_num_groups,
                              scaling_factor=c.scaling_factor, shift_factor=c.shift_factor)
        for i, v in enumerate(c.block_out_channels):
            cfg.block_out_channels[i] = int(v)
        ctx = L.vp()
        L.check(lib.tpdm_vae_create(C.byref(cfg), C.byref(ctx)))
        self._ctx = ctx
        self.repack()

    def repack(self) -> None:
        """(re)builds the packed bf16 / fp32 device copies the library reads; call after changing parameters"""
        if self._ctx is None:
            return self._ensure_ctx()
        lib = L.load()
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("tpdm_b200 AutoencoderKL needs its parameters on a CUDA device (there is no CPU path)")
        keep: List[torch.Tensor] = []

        def hold(t: torch.Tensor) -> int:
            keep.append(t)
            return t.data_ptr()

        d = self.decoder
        resnets = list(d.mid_block.resnets) + [r for b in d.up_blocks for r in b.resnets]
        arr = (L.TpdmVaeResnet * len(resnets))()
        for i, r in enumerate(resnets):
            a = arr[i]
            a.norm1_w, a.norm1_b = hold(_f32(r.norm1.weight, dev)), hold(_f32(r.norm1.bias, dev))
            a.conv1_w, a.conv1_b = hold(_conv_w(r.conv1, dev)), hold(_f32(r.conv1.bias, dev))
            a.norm2_w, a.norm2_b = hold(_f32(r.norm2.weight, dev)), hold(_f32(r.norm2.bias, dev))
            a.conv2_w, a.conv2_b = hold(_conv_w(r.conv2, dev)), hold(_f32(r.conv2.bias, dev))
            if hasattr(r, "conv_shortcut"):
                sw = r.conv_shortcut.weight.detach().to(dev, torch.float32).reshape(r.conv_shortcut.weight.shape[0], -1)
                a.short_w, a.short_b = hold(sw.to(torch.bfloat16).contiguous()), hold(_f32(r.conv_shortcut.bias, dev))
        w = L.TpdmVaeWeights()
        w.conv_in_w, w.conv_in_b = hold(_conv_w(d.conv_in, dev, pad_in=64)), hold(_f32(d.conv_in.bias, dev))
        w.resnets, w.n_resnets = arr, len(resnets)
        at = d.mid_block.attentions[0]
        w.attn_norm_w, w.attn_norm_b = hold(_f32(at.group_norm.weight, dev)), hold(_f32(at.group_norm.bias, dev))
        lin = lambda m: hold(m.weight.detach().to(dev, torch.bfloat16).contiguous())
        w.attn_q_w, w.attn_k_w, w.attn_v_w, w.attn_o_w = lin(at.to_q), lin(at.to_k), lin(at.to_v), lin(at.to_out[0])
        w.attn_q_b, w.attn_k_b = hold(_f32(at.to_q.bias, dev)), hold(_f32(at.to_k.bias, dev))
        w.attn_v_b, w.attn_o_b = hold(_f32(at.to_v.bias, dev)), hold(_f32(at.to_out[0].bias, dev))
        ups = [b.upsamplers[0].conv for b in d.up_blocks if hasattr(b, "upsamplers")]
        upw, upb = (L.vp * max(len(ups), 1))(), (L.vp * max(len(ups), 1))()
        for i, cv in enumerate(ups):
            upw[i], upb[i] = hold(_conv_w(cv, dev)), hold(_f32(cv.bias, dev))
        w.up_conv_w, w.up_conv_b, w.n_upsamplers = upw, upb, len(ups)
        w.norm_out_w, w.norm_out_b = hold(_f32(d.conv_norm_out.weight, dev)), hold(_f32(d.conv_norm_out.bias, dev))
        w.conv_out_w, w.conv_out_b = hold(_conv_w(d.conv_out, dev, pad_out=8)), hold(_f32(d.conv_out.bias, dev, pad=8))
        with torch.cuda.device(dev):
            L.check(lib.tpdm_vae_set_weights(self._ctx, C.byref(w)))
        self._packed = keep

    def __del__(self):
        try:
            if getattr(self, "_ctx", None) is not None:
                L.load().tpdm_vae_destroy(self._ctx)
        except Exception:
            pass

    # ---- decode ------------------------------------------------------------------------------------------------
    @property
    def upscale(self) -> int:
        return 2 ** (len(self.config.block_out_channels) - 1)

    def _run(self, latents: torch.Tensor, apply_scaling: bool, want_image: bool, want_rgb: bool):
        if latents.dim() != 4 or latents.shape[1] != self.config.latent_channels:
            raise ValueError(f"expected latents of shape (B, {self.config.latent_channels}, h, w), got {tuple(latents.shape)}")
        self._ensure_ctx()
        lib = L.load()
        dev = self.device
        x = latents.to(device=dev, dtype=torch.float32).contiguous()
        B, _, h, w = x.shape
        nbytes = lib.tpdm_vae_workspace_bytes(self._ctx, h, w)
        if self._workspace is None or self._workspace.numel() < nbytes + 1024:
            self._workspace = None
            self._workspace, self._workspace_base = L.aligned_workspace(nbytes, dev)
        base = self._workspace_base
        H, W = h * self.upscale, w * self.upscale
        image = torch.empty(B, self.config.out_channels, H, W, device=dev) if want_image else None
        rgb = torch.empty(B, H, W, self.config.out_channels, device=dev, dtype=torch.uint8) if want_rgb else None
        with torch.cuda.device(dev):
            L.check(lib.tpdm_vae_decode(self._ctx, L.ptr(x), 1 if apply_scaling else 0, B, h, w, base, nbytes, L.ptr(image), L.ptr(rgb),
                                        torch.cuda.current_stream().cuda_stream))
        return image, rgb

    def decode(self, z: torch.Tensor, return_dict: bool = True, generator=None):
        """``AutoencoderKL.decode``: z (already un-scaled) -> image (B, 3, 8h, 8w) in the parameter dtype."""
        image, _ = self._run(z, False, True, False)
        image = image.to(self.dtype)
        return SimpleNamespace(sample=image) if return_dict else (image,)

    def decode_latents(self, latents: torch.Tensor, output_type: str = "pt"):
        """The reference's whole tail in one call (modeling_sd3_pnt.py:653-655): un-scale, decode, and for ``"uint8"`` /
        ``"pil"`` the VaeImageProcessor post-processing on the device.  ``"pt"`` -> fp32 image (B, 3, H, W);
        ``"uint8"`` -> (B, H, W, 3) uint8 on the device; ``"pil"`` -> list of PIL images."""
        if output_type == "pt":
            return self._run(latents, True, True, False)[0]
        _, rgb = self._run(latents, True, False, True)
        if output_type == "uint8":
            return rgb
        if output_type == "pil":
            from PIL import Image
            return [Image.fromarray(a) for a in rgb.cpu().numpy()]
        raise ValueError(f"unknown output_type {output_type!r}")
