"""Element-by-element check of the joint attention kernel against a float64 reference, plus a gain check and a check that the
launch wrote nothing outside the rows it owns (tests/kernel_check.py does the same for the GEMMs).

For one (batch b, head h) the reference is s = q k^T / sqrt(d), P = softmax(s), ref = P v, all in float64 from the same bf16
inputs the kernel reads.  Every element of O gets its own bound

    |out - ref| <= TAU_ATTN * M + 2^-8 |ref|,    M_i = sum_j P_ij |v_j|

M is the scale of the error the kernel makes by rounding P to bf16 (unit roundoff 2^-8) for P V while the row sum l adds the
unrounded fp32 p: errors common to every key of a row (the reference m_ref, the power-of-two rescales of the row-sum guard)
cancel in 1 / l.  2^-8 |ref| is the bf16 rounding of the output.  Pad columns [d, dp) have ref = M = 0 and must be exactly 0.

Rounding of the fp32 scores would add 2^-15 sum_j P_ij |v_j| A_ij with A_ij = |q_i| |k_j| / sqrt(d).  The term is computed and its
ratio printed beside the plain one, but the bound leaves it out (USE_SCORE_TERM): on a B200 the +-1e4-logit tests stay at 2.1e-3
without it (1.5e-3 with it), inside TAU_ATTN.

The element bound cannot see a small one-sided error: P packed by truncation instead of round-to-nearest stays below it while
it scales every output by about (1 - 2^-9).  So the fitted gain beta = sum (out - ref) ref / sum ref^2 must also satisfy
|beta| <= GAIN_TOL, over the whole launch and over every (b, h) slice of at least 128 query rows.  beta is not free of noise even
when the kernel rounds to nearest: the rounding of a row's few dominant P_ij is shared by all d columns of that row, so a slice
averages over its rows, not its elements (about 1e-4 standard deviation at 128 rows; the CPU emulation of the kernel with
round-to-nearest P reaches 2.5e-4 on the 300-row slices of test_joint_attention[2-300-3-32-0], and the B200 2.7e-4 there).

TAU_ATTN and GAIN_TOL are the smallest powers of two at least twice the largest value observed on a B200 over the attention
tests (tests/test_attention_elementwise_gpu.py and the attention tests of tests/test_parity_gpu.py).
"""
from __future__ import annotations

import math

import torch

from kernel_check import assert_launch, bits, guarded, ratio

# Largest observed ratio on a B200 (1000 W power limit): 3.73e-3, test_adversarial_masking[129-64-deep] (2.4e-3 on random
# inputs); 2 * 3.73e-3 = 7.5e-3 <= 2^-7 = 7.8e-3.
TAU_ATTN = 2.0 ** -7
# Largest observed |beta| on a B200 (1000 W power limit): 2.72e-4, one (b, h) slice of test_joint_attention[2-300-3-32-0]; the
# largest over a whole launch was 1.4e-4 (S = 2, eight rows).  2 * 2.72e-4 = 5.4e-4 <= 2^-10 = 9.8e-4.  P packed by truncation
# gives |beta| 2.0e-3 to 2.9e-3 on the same tests.
GAIN_TOL = 2.0 ** -10
GAIN_MIN_ROWS = 128
SCORE_ROUNDING = 2.0 ** -15
USE_SCORE_TERM = False

LOG2E = 1.4426950408889634
Q_TILE = 128


def owned_rows(S: int, q_rows: int = 0) -> int:
    """Rows of every batch entry the kernel stores: the query tiles that q_rows selects (all when 0), rows >= S never."""
    if q_rows <= 0 or q_rows >= S:
        return S
    return min(S, Q_TILE * math.ceil(q_rows / Q_TILE))


def attention_reference(qkv: torch.Tensor, d: int, rows: int | None = None, block_elems: int = 1 << 25):
    """qkv [Bt][S][3][H][dp] (bf16) -> (ref, M, A) float64 [Bt][rows][H][d] for the first `rows` queries of every (b, h):
    ref = softmax(q k^T / sqrt(d)) v, M = P |v| and the score-rounding scale A = sum_j P_ij |v_j| |q_i| |k_j| / sqrt(d).
    Computed on qkv's device in blocks of query rows and slices of at most block_elems scores."""
    Bt, S, _, H, _ = qkv.shape
    R = S if rows is None else rows

    def part(i, n):
        return qkv[:, :n, i, :, :d].permute(0, 2, 1, 3).reshape(Bt * H, n, d).double()

    q, k, v = part(0, R), part(1, S), part(2, S)
    inv = 1.0 / math.sqrt(d)
    va = v.abs()
    vak = va * k.norm(dim=-1, keepdim=True)
    qn = q.norm(dim=-1, keepdim=True) * inv
    ref, mag, sc = (torch.empty(Bt * H, R, d, dtype=torch.float64, device=qkv.device) for _ in range(3))
    c = max(1, min(R, block_elems // S))
    g = max(1, block_elems // (c * S))
    for g0 in range(0, Bt * H, g):
        g1 = min(Bt * H, g0 + g)
        kt = k[g0:g1].transpose(-1, -2)
        for r0 in range(0, R, c):
            r1 = min(R, r0 + c)
            p = q[g0:g1, r0:r1] @ kt
            p.mul_(inv)
            p.sub_(p.amax(-1, keepdim=True)).exp_()
            p.div_(p.sum(-1, keepdim=True))
            ref[g0:g1, r0:r1] = p @ v[g0:g1]
            mag[g0:g1, r0:r1] = p @ va[g0:g1]
            sc[g0:g1, r0:r1] = (p @ vak[g0:g1]) * qn[g0:g1, r0:r1]
    back = lambda t: t.view(Bt, H, R, d).permute(0, 2, 1, 3)
    return back(ref), back(mag), back(sc)


def attention_out(Bt: int, S: int, H: int, dp: int, device="cuda"):
    """(buf, out): the sentinel-guarded output of one launch, out [Bt][S][H][dp] bf16 with one whole query tile of guard rows
    (128 * H * dp elements) before and after it."""
    buf, out = guarded((Bt, S, H, dp), torch.bfloat16, device=device, pad=Q_TILE * H * dp)
    return buf, out


def launch_attention(L, qkv: torch.Tensor, d: int, q_rows: int = 0):
    """One tpdm_joint_attention launch into a fresh guarded output: (buf, before, out).  qkv must come back bit-identical."""
    Bt, S, _, H, dp = qkv.shape
    buf, out = attention_out(Bt, S, H, dp, device=qkv.device)
    before = buf.clone()
    qkv_before = qkv.clone()
    L.check(L.load().tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, dp, d, q_rows, None))
    torch.cuda.synchronize()
    assert torch.equal(bits(qkv), bits(qkv_before)), "the launch changed its input"
    return buf, before, out


def attention_gain(out: torch.Tensor, ref: torch.Tensor):
    """beta = sum (out - ref) ref / sum ref^2 over the whole tensor and per (b, h) slice: (whole, [Bt][H])."""
    o, r = out.double(), ref.double()
    num = ((o - r) * r).sum(dim=(1, 3))
    den = (r * r).sum(dim=(1, 3))
    whole = float(num.sum() / den.sum()) if float(den.sum()) > 0 else 0.0
    per = torch.where(den > 0, num / den.clamp_min(1e-300), torch.zeros_like(num))
    return whole, per


def assert_gain(out: torch.Tensor, ref: torch.Tensor, gain_tol: float = GAIN_TOL, what: str = "") -> float:
    """|beta| <= gain_tol over the whole launch and over every (b, h) slice of >= GAIN_MIN_ROWS query rows; returns the largest."""
    whole, per = attention_gain(out, ref)
    worst = abs(whole)
    if out.shape[1] >= GAIN_MIN_ROWS:
        worst = max(worst, float(per.abs().max()))
    print(f"[attention_check] {what} gain: whole launch {whole:+.3e}, largest |beta| {worst:.3e} (tol {gain_tol:.3e})")
    if out.shape[1] >= GAIN_MIN_ROWS and not float(per.abs().max()) <= gain_tol:
        b, h = (int(i) for i in torch.unravel_index(per.abs().argmax(), per.shape))
        raise AssertionError(f"{what}: gain of (b {b}, h {h}) {float(per[b, h]):+.3e} outside +-{gain_tol:.3e} "
                             f"({int((per.abs() > gain_tol).sum())} of {per.numel()} slices)")
    if not abs(whole) <= gain_tol:
        raise AssertionError(f"{what}: gain of the whole launch {whole:+.3e} outside +-{gain_tol:.3e}")
    return worst


def assert_attention(buf, before, out, qkv, d: int, q_rows: int = 0, what: str = "", tau: float = TAU_ATTN,
                     gain_tol: float | None = GAIN_TOL) -> dict:
    """Checks one launch: every owned element (rows [0, owned_rows) of every batch entry, all dp columns) within its bound, pad
    columns exactly 0, everything else of buf bit-identical to `before`, and the gain.  Returns the observed maxima.
    gain_tol None skips the gain, for inputs whose rows are near copies of one vector (one key dominating every row): their
    output roundings do not average out, and beta measures the rounding of that one vector."""
    Bt, S, H, dp = out.shape
    R = owned_rows(S, q_rows)
    ref, mag, sc = attention_reference(qkv, d, R)
    full = lambda t: torch.nn.functional.pad(t, (0, dp - d))
    region = out[:, :R]
    fref, fmag, fsc = full(ref), full(mag), full(sc)
    plain = float(ratio(region, fref, fmag).max())
    scored = float(ratio(region, fref, fmag + SCORE_ROUNDING * fsc).max())
    print(f"[attention_check] {what} max ratio {plain:.3e}, with the score term {scored:.3e} (tau {tau:.3e})")
    assert_launch(buf, before, [(region, fref, fmag + SCORE_ROUNDING * fsc if USE_SCORE_TERM else fmag, None)], tau, what)
    gain = assert_gain(region[..., :d], ref, gain_tol, what) if gain_tol is not None else None
    return {"ratio": plain, "ratio_score": scored, "gain": gain}


def check_attention(L, qkv: torch.Tensor, d: int, q_rows: int = 0, what: str = "", gain_tol: float | None = GAIN_TOL) -> dict:
    """launch_attention + assert_attention."""
    buf, before, out = launch_attention(L, qkv, d, q_rows)
    return assert_attention(buf, before, out, qkv, d, q_rows, what, gain_tol=gain_tol)


def adversarial_qkv(Bt: int, S: int, H: int, d: int, dp: int, lo: float, hi: float, generator=None, device="cuda"):
    """Inputs under which a masking error is gross: every score lies about lo..hi log2 units below 0 (lo < hi < 0; keys point
    away from the queries), so a zero-filled key past S (score 0) would outweigh the whole row, and a first-tile maximum taken
    over such a key would underflow every real p.  The last key, the single valid key of the last tile when S % 128 == 1,
    carries the largest score of every row, so a mask one key too wide is gross too.  V is random."""
    scale = LOG2E / math.sqrt(d)
    a_lo, a_hi = math.sqrt(-hi / scale), math.sqrt(-lo / scale)
    e = torch.randn(d, generator=generator)
    e /= e.norm()
    a = a_lo + (a_hi - a_lo) * torch.rand(Bt, S, H, 1, generator=generator)
    b = a_lo + (a_hi - a_lo) * torch.rand(Bt, S, H, 1, generator=generator)
    b[:, S - 1] = 0.85 * a_lo
    qkv = torch.zeros(Bt, S, 3, H, dp)
    qkv[:, :, 0, :, :d] = a * e + 0.3 * torch.randn(Bt, S, H, d, generator=generator)
    qkv[:, :, 1, :, :d] = -b * e + 0.3 * torch.randn(Bt, S, H, d, generator=generator)
    qkv[:, :, 2, :, :d] = torch.randn(Bt, S, H, d, generator=generator)
    return qkv.bfloat16().to(device).contiguous()
