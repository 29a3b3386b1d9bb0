"""Drop-in for /root/reference/src/models/stable_diffusion_3/transformer_sd3.py.

``CustomSD3Transformer2DModel`` keeps the reference's constructor kwargs (transformer_sd3.py:91-108), ``.config``
attribute access, diffusers state-dict names (SURVEY.md section 8b) and the 4-tuple / output-dataclass return of
``forward`` (:401-409).  The modules below only HOLD parameters; ``forward`` runs in libtpdm_b200.so.
"""
from __future__ import annotations

from dataclasses import dataclass, fields
from types import SimpleNamespace
from typing import List, Optional, Tuple, Union

import numpy as np
import torch
import torch.nn as nn

from .engine import Engine, check_mmdit_precision


class BaseOutput(dict):
    """Minimal stand-in for diffusers.utils.BaseOutput: dataclass fields readable as attributes, keys and by index."""

    def __post_init__(self):
        for f in fields(self):
            v = getattr(self, f.name)
            if v is not None:
                dict.__setitem__(self, f.name, v)

    def __getitem__(self, k):
        if isinstance(k, str):
            return dict.__getitem__(self, k)
        return self.to_tuple()[k]

    def __setattr__(self, name, value):
        if name in self.keys() and value is not None:
            dict.__setitem__(self, name, value)
        object.__setattr__(self, name, value)

    def __setitem__(self, key, value):
        dict.__setitem__(self, key, value)
        object.__setattr__(self, key, value)

    def to_tuple(self):
        return tuple(self[k] for k in self.keys())


@dataclass
class CustomTransformer2DModelOutput(BaseOutput):
    """transformer_sd3.py:46-64."""

    sample: "torch.Tensor"
    temb: Optional[torch.Tensor] = None
    hidden_states_1: Optional[torch.Tensor] = None
    hidden_states_2: Optional[torch.Tensor] = None


# ---- parameter containers with the diffusers attribute names ---------------------------------------------------
def _sincos_table(embed_dim: int, grid_size: int, base_size: int) -> torch.Tensor:
    """diffusers get_2d_sincos_pos_embed(embed_dim, grid_size, base_size=base_size): float64 math, MAE layout
    (first half of the channels encodes the column coordinate)."""
    def one_d(dim, pos):
        omega = np.arange(dim // 2, dtype=np.float64) / (dim / 2.0)
        omega = 1.0 / 10000 ** omega
        out = np.einsum("m,d->md", pos.reshape(-1), omega)
        return np.concatenate([np.sin(out), np.cos(out)], axis=1)

    coords = np.arange(grid_size, dtype=np.float32) / (grid_size / base_size)
    grid = np.stack(np.meshgrid(coords, coords), axis=0).reshape([2, 1, grid_size, grid_size])
    table = np.concatenate([one_d(embed_dim // 2, grid[0]), one_d(embed_dim // 2, grid[1])], axis=1)
    return torch.from_numpy(table).float().unsqueeze(0)


class _PatchEmbed(nn.Module):
    def __init__(self, sample_size, patch_size, in_channels, embed_dim, pos_embed_max_size, **fk):
        super().__init__()
        self.proj = nn.Conv2d(in_channels, embed_dim, kernel_size=(patch_size, patch_size), stride=patch_size, bias=True, **fk)
        table = _sincos_table(embed_dim, pos_embed_max_size, sample_size // patch_size)
        self.register_buffer("pos_embed", table.to(device=fk.get("device")), persistent=True)


class _TwoLayer(nn.Module):
    def __init__(self, d_in, d, **fk):
        super().__init__()
        self.linear_1 = nn.Linear(d_in, d, **fk)
        self.linear_2 = nn.Linear(d, d, **fk)


class _TimeTextEmbed(nn.Module):
    def __init__(self, d, pooled, **fk):
        super().__init__()
        self.timestep_embedder = _TwoLayer(256, d, **fk)
        self.text_embedder = _TwoLayer(pooled, d, **fk)


class _AdaNorm(nn.Module):
    def __init__(self, d, mult, **fk):
        super().__init__()
        self.linear = nn.Linear(d, mult * d, **fk)


class _RMSWeight(nn.Module):
    def __init__(self, d, **fk):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(d, **fk))


class _Attention(nn.Module):
    def __init__(self, d, dim_head, context_pre_only, qk_norm, **fk):
        super().__init__()
        for n in ("to_q", "to_k", "to_v", "add_k_proj", "add_v_proj", "add_q_proj"):
            setattr(self, n, nn.Linear(d, d, **fk))
        self.to_out = nn.ModuleList([nn.Linear(d, d, **fk), nn.Identity()])
        if not context_pre_only:
            self.to_add_out = nn.Linear(d, d, **fk)
        if qk_norm == "rms_norm":
            for n in ("norm_q", "norm_k", "norm_added_q", "norm_added_k"):
                setattr(self, n, _RMSWeight(dim_head, **fk))


class _GELUProj(nn.Module):
    def __init__(self, d, **fk):
        super().__init__()
        self.proj = nn.Linear(d, 4 * d, **fk)


class _FeedForward(nn.Module):
    def __init__(self, d, **fk):
        super().__init__()
        self.net = nn.ModuleList([_GELUProj(d, **fk), nn.Identity(), nn.Linear(4 * d, d, **fk)])


class _SelfAttention(nn.Module):
    """parameter holder of attn2 in an SD3.5 dual-attention block"""

    def __init__(self, d, dim_head, qk_norm, **fk):
        super().__init__()
        for n in ("to_q", "to_k", "to_v"):
            setattr(self, n, nn.Linear(d, d, **fk))
        self.to_out = nn.ModuleList([nn.Linear(d, d, **fk), nn.Identity()])
        if qk_norm == "rms_norm":
            for n in ("norm_q", "norm_k"):
                setattr(self, n, _RMSWeight(dim_head, **fk))


class _JointBlock(nn.Module):
    def __init__(self, d, dim_head, context_pre_only, qk_norm, use_dual_attention=False, **fk):
        super().__init__()
        self.context_pre_only = context_pre_only
        self.use_dual_attention = use_dual_attention
        self.norm1 = _AdaNorm(d, 9 if use_dual_attention else 6, **fk)   # SD35AdaLayerNormZeroX : AdaLayerNormZero
        self.norm1_context = _AdaNorm(d, 2 if context_pre_only else 6, **fk)
        self.attn = _Attention(d, dim_head, context_pre_only, qk_norm, **fk)
        if use_dual_attention:
            self.attn2 = _SelfAttention(d, dim_head, qk_norm, **fk)
        self.ff = _FeedForward(d, **fk)
        if not context_pre_only:
            self.ff_context = _FeedForward(d, **fk)


class CustomSD3Transformer2DModel(nn.Module):
    """The SD3 MMDiT that additionally returns temb and the first / last hidden states (TPM taps)."""

    def __init__(
        self,
        sample_size: int = 128,
        patch_size: int = 2,
        in_channels: int = 16,
        num_layers: int = 18,
        attention_head_dim: int = 64,
        num_attention_heads: int = 18,
        joint_attention_dim: int = 4096,
        caption_projection_dim: int = 1152,
        pooled_projection_dim: int = 2048,
        out_channels: int = 16,
        pos_embed_max_size: int = 96,
        dual_attention_layers: Tuple[int, ...] = (),
        qk_norm: Optional[str] = None,
        device=None,
        dtype=None,
        mmdit_precision: str = "bf16",
    ):
        """``mmdit_precision``: ``"bf16"`` (default) or ``"fp8"``, which runs the QKV and FF1 projections of both streams as
        E4M3 GEMMs with per-token activation and per-channel weight scales (INTEGRATION.md states the accuracy); the
        attribute of the same name may be changed later, the next forward then builds a matching engine."""
        super().__init__()
        self.mmdit_precision = mmdit_precision
        dual_attention_layers = tuple(int(i) for i in dual_attention_layers)
        if any(i < 0 or i >= num_layers or i >= 64 for i in dual_attention_layers):
            raise ValueError(f"dual_attention_layers {dual_attention_layers} must name layers below min(num_layers, 64)")
        if qk_norm not in (None, "rms_norm"):
            raise ValueError(f"unknown qk_norm: {qk_norm}")
        self.config = SimpleNamespace(
            sample_size=sample_size, patch_size=patch_size, in_channels=in_channels, num_layers=num_layers,
            attention_head_dim=attention_head_dim, num_attention_heads=num_attention_heads, joint_attention_dim=joint_attention_dim,
            caption_projection_dim=caption_projection_dim, pooled_projection_dim=pooled_projection_dim,
            out_channels=out_channels if out_channels is not None else in_channels, pos_embed_max_size=pos_embed_max_size,
            dual_attention_layers=tuple(dual_attention_layers), qk_norm=qk_norm)
        self.out_channels = self.config.out_channels
        self.inner_dim = num_attention_heads * attention_head_dim
        if self.inner_dim != caption_projection_dim:
            raise ValueError("num_attention_heads * attention_head_dim must equal caption_projection_dim")
        fk = {"device": device, "dtype": dtype}
        d = self.inner_dim
        self.pos_embed = _PatchEmbed(sample_size, patch_size, in_channels, d, pos_embed_max_size, **fk)
        self.time_text_embed = _TimeTextEmbed(d, pooled_projection_dim, **fk)
        self.context_embedder = nn.Linear(joint_attention_dim, caption_projection_dim, **fk)
        self.transformer_blocks = nn.ModuleList(
            [_JointBlock(d, attention_head_dim, i == num_layers - 1, qk_norm, use_dual_attention=i in dual_attention_layers, **fk)
             for i in range(num_layers)])
        self.norm_out = _AdaNorm(d, 2, **fk)
        self.proj_out = nn.Linear(d, patch_size * patch_size * self.out_channels, bias=True, **fk)
        self.gradient_checkpointing = False
        self._engine: Optional[Engine] = None
        self._engine_key = None

    @property
    def mmdit_precision(self) -> str:
        return self._mmdit_precision

    @mmdit_precision.setter
    def mmdit_precision(self, value: str) -> None:
        self._mmdit_precision = check_mmdit_precision(value)

    # -- engine management: repack whenever a parameter tensor was replaced / modified in place ---------------------
    def _weights_key(self):
        return tuple((p.data_ptr(), p._version, p.device) for p in list(self.parameters()) + list(self.buffers()))

    def engine_config(self) -> dict:
        c = self.config
        return dict(num_layers=c.num_layers, num_attention_heads=c.num_attention_heads, attention_head_dim=c.attention_head_dim,
                    joint_attention_dim=c.joint_attention_dim, pooled_projection_dim=c.pooled_projection_dim,
                    in_channels=c.in_channels, out_channels=c.out_channels, patch_size=c.patch_size,
                    pos_embed_max_size=c.pos_embed_max_size, qk_norm=c.qk_norm, dual_attention_layers=c.dual_attention_layers)

    def get_engine(self) -> Engine:
        key = (self._weights_key(), self.mmdit_precision)
        if self._engine is None or key != self._engine_key:
            dev = self.proj_out.weight.device
            self._engine = Engine(self.engine_config(), dev, transformer_sd=self.state_dict(), transformer_cfg=self.config,
                                  mmdit_precision=self.mmdit_precision)
            self._engine_key = key
        return self._engine

    @property
    def device(self):
        return self.proj_out.weight.device

    @property
    def dtype(self):
        return self.proj_out.weight.dtype

    @torch.no_grad()
    def forward(
        self,
        hidden_states: torch.FloatTensor,
        encoder_hidden_states: torch.FloatTensor = None,
        pooled_projections: torch.FloatTensor = None,
        timestep: torch.LongTensor = None,
        block_controlnet_hidden_states: List = None,
        return_dict: bool = True,
    ) -> Union[Tuple, CustomTransformer2DModelOutput]:
        if block_controlnet_hidden_states is not None:
            raise ValueError("block_controlnet_hidden_states is not supported by tpdm_b200 (not on the TPDM path)")
        if encoder_hidden_states is None or pooled_projections is None or timestep is None:
            raise ValueError("encoder_hidden_states, pooled_projections and timestep are required")
        out_dtype = hidden_states.dtype
        output, temb, h1, h2 = self.get_engine().mmdit_forward(hidden_states, encoder_hidden_states, pooled_projections, timestep)
        output, temb, h1, h2 = (t.to(out_dtype) for t in (output, temb, h1, h2))
        if not return_dict:
            return (output, temb, h1, h2)
        return CustomTransformer2DModelOutput(sample=output, temb=temb, hidden_states_1=h1, hidden_states_2=h2)
