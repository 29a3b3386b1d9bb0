"""FP8 (E4M3) fake quantization for the tests of tpdm_b200's opt-in ``mmdit_precision="fp8"``: the rounding of
``tpdm_quantize_fp8_rows`` restated in torch, and a switch that applies it to the QKV and FF1 linears of both streams of the
fp32 oracle (``oracle.sd3_oracle.OracleSD3Transformer``) without changing its parameters or state-dict names."""
from typing import Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

E4M3_MAX = 448.0


def quantize_e4m3_rows(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per row of the last dim: amax = max |x|, codes = round-to-nearest-even E4M3 of x * (448 / amax), scale = amax / 448
    (fp32 divisions), so x ~= codes * scale.  A zero row gets scale 1 and zero codes.  -> (float8_e4m3fn codes, fp32 scales)."""
    x = x.float()
    amax = x.abs().amax(dim=-1, keepdim=True)
    nz = amax > 0
    inv = torch.where(nz, E4M3_MAX / amax, torch.ones_like(amax))
    scale = torch.where(nz, amax / E4M3_MAX, torch.ones_like(amax))
    return (x * inv).to(torch.float8_e4m3fn), scale.squeeze(-1)


def fake_quant_e4m3_rows(x: torch.Tensor) -> torch.Tensor:
    codes, scale = quantize_e4m3_rows(x)
    return codes.float() * scale.unsqueeze(-1)


class FakeQuantE4M3Linear(nn.Linear):
    """nn.Linear with per-token E4M3 activations and per-output-channel E4M3 weights, fp32 products and bias."""

    def forward(self, x):
        return F.linear(fake_quant_e4m3_rows(x), fake_quant_e4m3_rows(self.weight), self.bias)


def set_fp8_fake_quant(transformer: nn.Module, enabled: bool = True) -> nn.Module:
    """On an OracleSD3Transformer: switch the joint-attention QKV linears (image and text stream) and FF1 of both feed-forwards to FakeQuantE4M3Linear
    (``enabled``) or back to nn.Linear.  Parameters and state-dict names do not change; attn2, out-projections, FF2 and
    everything outside the blocks stay exact."""
    cls = FakeQuantE4M3Linear if enabled else nn.Linear
    for blk in transformer.transformer_blocks:
        a = blk.attn
        lins = [a.to_q, a.to_k, a.to_v, a.add_q_proj, a.add_k_proj, a.add_v_proj, blk.ff.net[0].proj]
        if not blk.context_pre_only:
            lins.append(blk.ff_context.net[0].proj)
        for lin in lins:
            lin.__class__ = cls
    return transformer
