"""CPU model of the fast attention kernel's softmax bookkeeping (tpdm_b200/csrc/attention_tcgen05.cu, the `tile` step of the fast
branch of attn_cta): two threads per query row, each over one 64-key half of every 128-key tile with its own partial row sum.  The
reference m_ref is the row maximum of the FIRST tile (both halves) and from then on it is guarded by the row sums at checkpoints,
every 4th tile: at checkpoint c both halves apply the total shift found in bump[c & 1] (O and l rescaled by that power of two),
and a half whose partial sum has passed 2^24 proposes its shift into bump[(c + 1) & 1], which takes effect at the next checkpoint.
A partial sum above 2^64 / inf / NaN, or an argument > 127 in a polynomial slot, flags the tile for the exact pass.  The model
mirrors that control flow in fp32 tile by tile and checks (i) that whenever no flag is raised the result equals softmax(S) V,
however the scores are ordered, and (ii) which growth the guard absorbs and which it flags.  No GPU, no library: this pins the
ALGORITHM; the kernel itself is compared with fp32 SDPA in tests/test_parity_gpu.py."""
import math

import pytest
import torch

KT, HALF = 128, 64
PROPOSE, HARD, POLY_MAX = 2.0 ** 24, 2.0 ** 64, 127.0
POLY = (torch.arange(HALF) // 2) % 4 == 3      # columns of a half whose pair of exponentials runs through the polynomial
SCALE = 1.4427 / 8


def guarded_softmax_v(scores: torch.Tensor, v: torch.Tensor, scale_log2: float):
    """scores [rows, S] fp32 (raw q.k), v [S, d].  Returns (out [rows, d], flagged: bool, moves: int), moves = reference shifts
    applied, summed over the rows."""
    rows, S = scores.shape
    n_kv = (S + KT - 1) // KT
    x_all = torch.full((rows, n_kv * KT), -math.inf)                 # keys >= S of the tail tile are masked to -inf
    x_all[:, :S] = scores.float() * scale_log2
    v_all = torch.zeros(n_kv * KT, v.shape[1])
    v_all[:S] = v.float()
    m_ref = x_all[:, :KT].max(dim=1).values                         # row maximum of the first key tile, both halves
    l = torch.zeros(rows, 2)                                         # partial row sum of each half
    pmax = torch.full((rows, 2), -math.inf)                          # running, never reset
    applied = torch.zeros(rows)                                      # total shift applied to the reference (same in both halves)
    bump = torch.zeros(2, rows)                                      # proposed totals, only ever raised
    o = torch.zeros(rows, v.shape[1])
    hard = torch.zeros(rows, dtype=torch.bool)
    moves = 0
    for j in range(n_kv):
        hard |= (pmax > POLY_MAX).any(dim=1)
        if j & 3 == 3:                                               # checkpoint c: apply bump[c & 1], propose into bump[(c + 1) & 1]
            c = j >> 2
            total = bump[c & 1].clone()
            e = torch.where(total > applied, total - applied, torch.zeros(rows))
            over = ~(l <= PROPOSE)
            hard |= (~(l <= HARD)).any(dim=1)
            floor_log2 = (torch.frexp(l).exponent - 1).float()
            shift = torch.maximum(total, applied)[:, None] + (floor_log2 - e[:, None]).clamp_min(0.0)
            proposal = torch.where(over & (l <= HARD), shift, torch.zeros(rows, 2)).max(dim=1).values
            bump[(c + 1) & 1] = torch.maximum(bump[(c + 1) & 1], proposal)
            alpha = torch.exp2(-e)
            m_ref = m_ref + e
            applied = torch.maximum(total, applied)
            l = l * alpha[:, None]
            o = o * alpha[:, None]
            moves += int((e > 0).sum())
        x = (x_all[:, j * KT:(j + 1) * KT] - m_ref[:, None]).view(rows, 2, HALF)
        pmax = torch.maximum(pmax, x[:, :, POLY].amax(dim=2))
        p = torch.exp2(x)                                            # fp32: overflows to inf above 128
        l = l + p.sum(dim=2)
        o = o + p.reshape(rows, KT).to(torch.bfloat16).float() @ v_all[j * KT:(j + 1) * KT]
    hard |= (~(l <= HARD)).any(dim=1) | (pmax > POLY_MAX).any(dim=1)
    return o / l.sum(dim=1)[:, None], bool(hard.any()), moves


def reference(scores, v, scale_log2):
    return torch.softmax(scores.double() * scale_log2 * math.log(2.0), dim=1) @ v.double()


def max_err(out, scores, v):
    return float((out.double() - reference(scores, v, SCALE)).abs().max())


@pytest.mark.parametrize("order", ["random", "ascending", "descending"])
def test_ordinary_scores_need_no_renormalisation(order):
    g = torch.Generator().manual_seed(0)
    s = torch.randn(64, 1000, generator=g) * 20.0
    if order != "random":
        s = s.sort(dim=1, descending=(order == "descending")).values
    v = torch.randn(1000, 16, generator=g)
    out, hard, n = guarded_softmax_v(s, v, SCALE)
    assert not hard
    if order != "ascending":
        assert n == 0
    assert max_err(out, s, v) < 2e-2


def growing_scores(log2_per_tile, n_tiles=16, seed=1):
    g = torch.Generator().manual_seed(seed)
    S = n_tiles * KT
    ramp = torch.arange(S).float() / KT * log2_per_tile / SCALE
    return torch.randn(32, S, generator=g) * 4.0 + ramp[None, :], torch.randn(S, 8, generator=g)


def test_steadily_growing_scores_are_renormalised_in_place():
    """+5 log2 units per tile over 16 tiles: the checkpoints move the reference, nothing is flagged, the result stays exact.  A
    proposal takes effect up to 8 tiles after the sum started to grow, so from 6 units per tile on a partial sum passes 2^64 before
    the reference catches up, and the tile goes to the exact pass."""
    s, v = growing_scores(5.0)
    out, hard, n = guarded_softmax_v(s, v, SCALE)
    assert not hard and n > 0
    assert max_err(out, s, v) < 2e-2
    for log2_per_tile in (6.0, 40.0):
        s, v = growing_scores(log2_per_tile)
        assert guarded_softmax_v(s, v, SCALE)[1], log2_per_tile


@pytest.mark.parametrize("jump_log2", [70.0, 200.0, 1e4])
def test_a_jump_the_guard_cannot_absorb_is_flagged(jump_log2):
    """A score more than 2^64 above everything the row has seen (here in a later tile, in a MUFU slot and in a polynomial slot):
    l or the polynomial argument leaves the range -> the tile must be flagged (the kernel then reruns it with per-chunk maxima)."""
    g = torch.Generator().manual_seed(2)
    for col in (3 * KT + 5, 3 * KT + 7):                       # column 7 of a tile is a polynomial slot (every 4th pair)
        s = torch.randn(8, 5 * KT, generator=g)
        s[2, col] += jump_log2 / SCALE
        v = torch.randn(5 * KT, 8, generator=g)
        out, hard, _ = guarded_softmax_v(s, v, SCALE)
        assert hard


def test_thirty_bit_jumps_stay_inside_the_range():
    """Scores that jump by 2^30 every 4th tile never overflow and never need the exact pass: the reference follows one checkpoint
    later.  The same jump in every tile outruns the checkpoints and is flagged."""
    g = torch.Generator().manual_seed(3)
    S = 16 * KT
    base = torch.randn(16, S, generator=g)
    v = torch.randn(S, 8, generator=g)
    s = base.clone()
    for t in range(4, 16, 4):
        s[:, t * KT + 11] += t // 4 * 30.0 / SCALE
    out, hard, n = guarded_softmax_v(s, v, SCALE)
    assert not hard and n > 0
    assert max_err(out, s, v) < 2e-2
    s = base.clone()
    for t in range(1, 16):
        s[:, t * KT + 11] += t * 30.0 / SCALE
    assert guarded_softmax_v(s, v, SCALE)[1]


def test_unflagged_results_match_softmax():
    """The property the kernel relies on, over random lengths, growth rates, jumps and score scales: whenever the guard raises no
    flag, the result is softmax(S) V."""
    g = torch.Generator().manual_seed(4)
    unflagged = moved = 0
    for _ in range(40):
        S = int(torch.randint(1, 20 * KT, (1,), generator=g))
        s = torch.randn(8, S, generator=g) * float(torch.rand(1, generator=g)) * 40.0
        s += torch.arange(S).float() / KT * float(torch.rand(1, generator=g)) * 8.0 / SCALE
        for _ in range(int(torch.randint(0, 4, (1,), generator=g))):
            col = int(torch.randint(0, S, (1,), generator=g))
            s[:, col] += float(torch.rand(1, generator=g)) * 80.0 / SCALE
        v = torch.randn(S, 8, generator=g)
        out, hard, n = guarded_softmax_v(s, v, SCALE)
        if not hard:
            unflagged += 1
            moved += n > 0
            assert max_err(out, s, v) < 2e-2
    assert unflagged >= 10 and moved >= 3
