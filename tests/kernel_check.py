"""Element-by-element comparison of a kernel's output with a float64 reference, plus a check that the launch wrote nothing
outside the regions it owns.

A rel-L2 bar over millions of elements cannot see a wrong 8-column group or one wrong 32 x 32 block (both move the norm by
less than the bf16 rounding noise of the whole tensor), nor a store past a ragged tile into a neighbour's rows.  Here every
element gets its own bound

    |out - ref| <= TAU * M  (+ 2^-8 |ref| for a bf16 output)  (+ 2^-11 |x| for GELU-tanh of the pre-activation x)

with M = |A| . |W|^T + |bias| in float64 (for out += gate * (acc + bias): |gate| (|A| . |W|^T + |bias|) + |out before|), the
scale of the fp32 accumulation error of that element.  2^-8 |ref| is one round-to-nearest bf16 rounding; gelu_tanh evaluates
0.5 x (1 + tanh.approx.f32(z)), and tanh.approx.f32 is within 2^-10.987 of tanh, so 0.5 |x| 2^-10 covers it with margin.

TAU is the smallest power of two at least twice the largest ratio |out - ref| / M (after the two terms above) observed on a
B200 over the GEMM and conv tests (tests/test_parity_gpu.py, tests/test_fp8_gpu.py, tests/test_launch_guards_gpu.py).
"""
from __future__ import annotations

import torch

# Largest observed ratio on a B200 (1000 W power limit): 1.56e-6, the conv3x3 test at g = 64, C = 3072 (K = 27648); the
# largest GEMM ratio was 8.3e-7 (K = 6144, epi 3).  2 * 1.56e-6 = 3.1e-6 <= 2^-18 = 3.8e-6.
TAU = 2.0 ** -18

BF16_ROUNDING = 2.0 ** -8
GELU_TANH_APPROX = 0.5 * 2.0 ** -10

# Sentinels written over every byte a launch must not touch: NaN payloads, so that a stray read of one shows too.
SENTINEL_F32 = 0x7FBF7FBF       # one fp32 NaN, or two bf16 0x7FBF NaNs
SENTINEL_BF16 = 0x7FBF
SENTINEL_U8 = 0xBF

_BITS = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}


def bits(t: torch.Tensor) -> torch.Tensor:
    """The raw bit pattern of t as an integer tensor of the same element size."""
    return t.view(_BITS[t.element_size()])


def fill_sentinel(t: torch.Tensor) -> torch.Tensor:
    bits(t).fill_({1: SENTINEL_U8, 2: SENTINEL_BF16, 4: SENTINEL_F32}[t.element_size()])
    return t


def guarded(shape, dtype, device="cuda", pad: int = 4096):
    """(buf, view): a flat sentinel-filled allocation with `pad` guard elements before and after the contiguous `view` of
    `shape` it holds, so that a store past either end of the view shows in assert_launch."""
    n = 1
    for s in shape:
        n *= s
    buf = fill_sentinel(torch.empty(n + 2 * pad, dtype=dtype, device=device))
    return buf, buf[pad:pad + n].view(shape)


def gemm_magnitude(A: torch.Tensor, W: torch.Tensor, bias: torch.Tensor | None = None) -> torch.Tensor:
    """M = |A| . |W|^T + |bias| in float64 (A [..., K], W [N, K])."""
    m = A.double().abs() @ W.double().abs().t()
    return m + bias.double().abs() if bias is not None else m


def ratio(out: torch.Tensor, ref: torch.Tensor, mag: torch.Tensor, gelu_x: torch.Tensor | None = None) -> torch.Tensor:
    """Per element (|out - ref| - rounding terms) / M, float64; inf where out is not finite or the excess has no magnitude."""
    o = out.double()
    ref = ref.double()
    excess = (o - ref).abs()
    if out.dtype == torch.bfloat16:
        excess = excess - BF16_ROUNDING * ref.abs()
    if gelu_x is not None:
        excess = excess - GELU_TANH_APPROX * gelu_x.double().abs()
    excess = excess.clamp_min(0.0)
    r = torch.where(excess > 0, excess / mag.double(), torch.zeros_like(excess))
    return torch.where(torch.isfinite(o), r.nan_to_num(nan=float("inf")), torch.full_like(r, float("inf")))


def assert_close(out, ref, mag, gelu_x=None, tau: float = TAU, what: str = "") -> float:
    """Every element of out within its bound; returns the largest ratio (printed, for setting TAU)."""
    assert out.shape == ref.shape == mag.shape, (what, out.shape, ref.shape, mag.shape)
    r = ratio(out, ref, mag, gelu_x)
    worst = float(r.max()) if r.numel() else 0.0
    print(f"[kernel_check] {what} max ratio {worst:.3e} (tau {tau:.3e})")
    if not worst <= tau:
        bad = (r > tau).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} of {r.numel()} elements outside the bound, first at {i}: "
                             f"out {float(out[i])} ref {float(ref[i])} M {float(mag[i])} ratio {float(r[i]):.3e} > tau {tau:.3e}")
    return worst


def assert_launch(buf: torch.Tensor, before: torch.Tensor, writes, tau: float = TAU, what: str = "") -> float:
    """buf: a whole allocation after the launch, before: its contents before.  writes: (view of buf, ref, M, gelu_x or None) for
    every region the launch owns; each is checked with assert_close, and every element outside them must be bit-identical to
    `before` (the sentinel, or the prior residual).  Returns the largest ratio."""
    assert buf.is_contiguous() and before.shape == buf.shape and before.dtype == buf.dtype
    owned = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    worst = 0.0
    for k, (view, ref, mag, gelu_x) in enumerate(writes):
        assert view.untyped_storage().data_ptr() == buf.untyped_storage().data_ptr(), "a region must be a view of buf"
        owned.as_strided(view.shape, view.stride(), view.storage_offset() - buf.storage_offset()).fill_(True)
        worst = max(worst, assert_close(view, ref, mag, gelu_x, tau, f"{what} region {k}"))
    stray = (bits(buf) != bits(before)) & ~owned
    if bool(stray.any()):
        where = stray.nonzero()
        raise AssertionError(f"{what}: {where.shape[0]} elements outside the written regions changed, first at {tuple(where[0].tolist())}")
    return worst
