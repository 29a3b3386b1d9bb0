"""The joint attention kernel element by element against float64 (tests/attention_check.py): key-tile edges, masking under
adversarial scores, padded heads and the production shapes, every output guarded by sentinels."""
import pytest
import torch

from attention_check import adversarial_qkv, check_attention

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from tpdm_b200 import _lib

    _lib.load()
    return _lib


def _qkv(Bt, S, H, d, dp, seed, std=1.5, head_scales=False, positive_v=False):
    """bf16 [Bt][S][3][H][dp] with zero pads; head_scales: q, k and v of every (b, h) scaled by its own factor in [0.5, 1.5], so
    a CTA that reads another head or batch entry is off by far more than the bound."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(Bt, S, 3, H, d, device="cuda", generator=g) * std
    if positive_v:
        x[:, :, 2] = 1.0 + 0.1 * x[:, :, 2] / std
    if head_scales:
        x *= 0.5 + torch.rand(Bt, 1, 3, H, 1, device="cuda", generator=g)
    qkv = torch.zeros(Bt, S, 3, H, dp, device="cuda")
    qkv[..., :d] = x
    return qkv.bfloat16().contiguous()


def _assert_no_redo(L):
    # in-range scores never leave the fast softmax (the exact pass is for rows the row-sum guard cannot keep in range)
    assert L.load().tpdm_attention_redo_count() in (0, -1)


@pytest.mark.parametrize("S", [1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513])
def test_key_tile_edges(L, S):
    """S <= 64: keys [64, 128) of the first tile all masked; multiples of 128: the masked tail path with nothing to mask; 129, 257,
    513: one valid key in the last tile; 512 / 513: the last tile on and off a row-sum guard checkpoint (tile j & 3 == 3)."""
    qkv = _qkv(2, S, 2, 64, 64, seed=S)
    check_attention(L, qkv, 64, what=f"S={S}")
    _assert_no_redo(L)


@pytest.mark.parametrize("depth", ["deep", "shallow"])
@pytest.mark.parametrize("d", [64, 96])
@pytest.mark.parametrize("S", [1, 65, 129, 257])
def test_adversarial_masking(L, S, d, depth):
    """All scores 100-300 (deep) or 24-60 (shallow) log2 units below 0 and the last key the largest of every row: a zero-filled key
    past S left unmasked outweighs the row (deep: its exponential overflows and would send the CTA to the exact pass, which the
    redo count shows; shallow: the output collapses by 2^20 or more), a masked key in the first tile's maximum underflows every
    p, and one key masked too many drops the row's dominant key."""
    lo, hi = (-300.0, -100.0) if depth == "deep" else (-60.0, -24.0)
    dp = 64 if d <= 64 else 128
    qkv = adversarial_qkv(2, S, 2, d, dp, lo, hi, torch.Generator().manual_seed(1000 * d + S))
    check_attention(L, qkv, d, what=f"adversarial {depth} S={S} d={d}", gain_tol=None)
    _assert_no_redo(L)


@pytest.mark.parametrize("d", [32, 96, 128])
def test_padded_heads(L, d):
    """d = 32 (dp 64) and d = 96 (dp 128): pad columns [d, dp) come out as exact zeros from the zero pads of the input; d = 128 has
    no pad."""
    dp = 64 if d <= 64 else 128
    qkv = _qkv(2, 589, 3, d, dp, seed=d, head_scales=True)
    check_attention(L, qkv, d, what=f"d={d}")
    _assert_no_redo(L)


@pytest.mark.parametrize("Bt,S,H,q_rows", [
    (2, 1357, 24, 0),       # SD3-medium 512^2 with CFG
    (2, 4429, 24, 0),       # 1024^2
    (2, 4429, 24, 4096),    # the last block's image-query rows
    (2, 4429, 38, 0),       # SD3.5-large width
    (1, 16717, 2, 0),       # 2048^2: 131 key tiles, 32 guard checkpoints
    (64, 1357, 3, 0),       # many batch entries
])
def test_production_shapes(L, Bt, S, H, q_rows):
    qkv = _qkv(Bt, S, H, 64, 64, seed=S + H + Bt, head_scales=True)
    check_attention(L, qkv, 64, q_rows=q_rows, what=f"Bt={Bt} S={S} H={H} q_rows={q_rows}")
    _assert_no_redo(L)


def test_positive_values(L):
    """V = 1 + 0.1 randn: |ref| ~ M, where a gain error of the kernel is largest."""
    qkv = _qkv(2, 4429, 4, 64, 64, seed=7, positive_v=True)
    check_attention(L, qkv, 64, what="positive V")
    _assert_no_redo(L)
