"""CPU tests of the attention checker (tests/attention_check.py) on an emulation of the kernel's numerics: fp32 scores, the
first-tile maximum as reference, p = exp2(s log2e / sqrt(d) - m_ref) in fp32, P rounded to bf16 for P V while l sums the fp32 p,
the output rounded to bf16.  The emulation must pass; each fault below must be flagged, and the ones marked so would have
passed the rel-L2 < 6e-3 bar the attention tests used before."""
import math

import pytest
import torch

from attention_check import (GAIN_TOL, LOG2E, Q_TILE, TAU_ATTN, adversarial_qkv, assert_attention, attention_gain,
                             attention_out, attention_reference)
from kernel_check import bits

OLD_REL_TOL = 6e-3


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


def emulate(qkv, d, *, truncate_p=False, unmasked_tail_keys=0):
    """The kernel's fast softmax on the CPU: out [Bt][S][H][dp] bf16 (pad columns from the zero pads of V)."""
    Bt, S, _, H, dp = qkv.shape
    Sp = Q_TILE * math.ceil(S / Q_TILE)                   # keys >= S of the last tile are zero-filled by TMA
    x = torch.zeros(Bt, Sp, 3, H, dp)
    x[:, :S] = qkv.float()
    q, k, v = (x[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    s = q[:, :, :S] @ k.transpose(-1, -2)
    s = s.masked_fill(torch.arange(Sp) >= S + unmasked_tail_keys, float("-inf"))
    scale = torch.tensor(LOG2E / math.sqrt(d), dtype=torch.float32)
    m_ref = (s[..., :Q_TILE] * scale).amax(-1, keepdim=True)
    p = torch.exp2(s * scale - m_ref)
    if truncate_p:
        P = (p.view(torch.int32) & -65536).view(torch.float32).bfloat16()
    else:
        P = p.bfloat16()
    out = (P.float() @ v) * (1.0 / p.sum(-1, keepdim=True))
    return out.bfloat16().permute(0, 2, 1, 3).contiguous()


def _qkv(Bt, S, H, d, dp, seed=0):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.zeros(Bt, S, 3, H, dp)
    qkv[..., :d] = torch.randn(Bt, S, 3, H, d, generator=g) * 1.5
    return qkv.bfloat16()


def _store(out_emul):
    """The emulated output written into a fresh guarded buffer, as a launch would: (buf, before, out)."""
    Bt, S, H, dp = out_emul.shape
    buf, out = attention_out(Bt, S, H, dp, device="cpu")
    before = buf.clone()
    out.copy_(out_emul)
    return buf, before, out


@pytest.mark.parametrize("Bt,S,H,d,dp", [(1, 2, 2, 64, 64), (2, 65, 2, 32, 64), (2, 300, 2, 64, 64), (1, 1357, 2, 96, 128)])
def test_emulated_kernel_passes(Bt, S, H, d, dp):
    qkv = _qkv(Bt, S, H, d, dp)
    got = assert_attention(*_store(emulate(qkv, d)), qkv, d, what=f"emulation S={S}")
    assert got["ratio"] <= TAU_ATTN and got["gain"] <= GAIN_TOL


@pytest.mark.parametrize("lo,hi", [(-300.0, -100.0), (-60.0, -24.0)])
@pytest.mark.parametrize("S", [1, 65, 129, 257])
def test_emulated_kernel_passes_adversarial_masking_inputs(S, lo, hi):
    qkv = adversarial_qkv(2, S, 2, 64, 64, lo, hi, torch.Generator().manual_seed(S), device="cpu")
    ref = attention_reference(qkv, 64)[0]
    assert float(ref.abs().max()) > 0.5    # the rows are not all underflowed to nothing in the reference either
    assert_attention(*_store(emulate(qkv, 64)), qkv, 64, what=f"adversarial S={S}", gain_tol=None)


def test_truncated_p_is_flagged_by_the_gain_and_passes_the_old_bar():
    qkv = _qkv(2, 1357, 2, 64, 64)
    buf, before, out = _store(emulate(qkv, 64, truncate_p=True))
    ref = attention_reference(qkv, 64)[0]
    assert _rel(out, ref) < OLD_REL_TOL
    with pytest.raises(AssertionError, match="gain of"):
        assert_attention(buf, before, out, qkv, 64, what="truncated P")
    whole, _ = attention_gain(out[..., :64], ref)
    assert whole < -GAIN_TOL                # one-sided: every output a little too small


@pytest.mark.parametrize("S,lo,hi", [(65, -300.0, -100.0), (129, -60.0, -24.0), (257, -300.0, -100.0)])
def test_one_unmasked_tail_key_is_flagged(S, lo, hi):
    qkv = adversarial_qkv(1, S, 2, 64, 64, lo, hi, torch.Generator().manual_seed(S), device="cpu")
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_attention(*_store(emulate(qkv, 64, unmasked_tail_keys=1)), qkv, 64, what=f"unmasked key S={S}")


def test_one_softmax_warps_rows_scaled_by_1_01_is_flagged_and_passes_the_old_bar():
    """32 rows of one query tile (the rows of one softmax warp) of one head, 1 % too large: the element bound flags the elements
    where the 1 % adds to the kernel's own rounding."""
    qkv = _qkv(2, 300, 2, 64, 64)
    buf, before, out = _store(emulate(qkv, 64))
    out[1, 160:192, 1] = (out[1, 160:192, 1].double() * 1.01).bfloat16()
    ref = attention_reference(qkv, 64)[0]
    assert _rel(out[..., :64], ref) < OLD_REL_TOL
    with pytest.raises(AssertionError, match=r"outside the bound, first at \(1, 1[6-9]\d, 1, "):
        assert_attention(buf, before, out, qkv, 64, what="scaled rows")


def test_one_row_past_s_stored_is_flagged():
    qkv = _qkv(2, 300, 2, 64, 64)
    buf, before, out = _store(emulate(qkv, 64))
    n = out.numel()
    pad = (buf.numel() - n) // 2
    row = buf[pad + n: pad + n + 2 * 64]              # row S of the last batch entry: the first guard row behind the output
    row.copy_(out[1, -1].reshape(-1))
    with pytest.raises(AssertionError, match="outside the written regions"):
        assert_attention(buf, before, out, qkv, 64, what="row S stored")


def test_query_tiles_left_out_by_q_rows_must_stay_sentinel():
    qkv = _qkv(1, 300, 2, 64, 64)
    full = emulate(qkv, 64)
    buf, out = attention_out(1, 300, 2, 64, device="cpu")
    before = buf.clone()
    out[:, :128].copy_(full[:, :128])
    assert_attention(buf, before, out, qkv, 64, q_rows=100, what="q_rows 100")
    out[:, 128].copy_(full[:, 128])                     # one row of the next tile, which q_rows = 100 leaves out
    with pytest.raises(AssertionError, match="outside the written regions"):
        assert_attention(buf, before, out, qkv, 64, q_rows=100, what="q_rows 100, row 128 stored")


def test_one_pad_column_not_zero_is_flagged():
    qkv = _qkv(2, 129, 2, 96, 128)
    buf, before, out = _store(emulate(qkv, 96))
    assert bool((bits(out[..., 96:]) == 0).all())
    assert_attention(buf, before, out, qkv, 96, what="d 96")
    out[0, 5, 1, 100] = 2.0 ** -20
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_attention(buf, before, out, qkv, 96, what="pad column")


def test_reference_blocks_do_not_change_the_result():
    qkv = _qkv(2, 300, 3, 64, 64)
    whole = attention_reference(qkv, 64)
    blocked = attention_reference(qkv, 64, block_elems=300 * 7)
    for a, b in zip(whole, blocked):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-14)
    ref = torch.nn.functional.scaled_dot_product_attention(*(qkv[:, :, i, :, :64].double().transpose(1, 2) for i in range(3)))
    assert torch.allclose(whole[0], ref.transpose(1, 2), rtol=1e-10, atol=1e-12)
