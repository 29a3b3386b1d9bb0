"""LayerNorm-modulate element by element against float64 (kernel_check.ln_modulate_reference, bound TAU_LN * M + 2^-8 |ref|):
every route of the kernel (the bulk-copy kernel at D = 1536, the register kernel at D = 384, the generic one at other widths),
ragged 32-row blocks, and the two-segment launch the MMDiT blocks run for their image and text rows."""
import pytest
import torch

from kernel_check import TAU_LN, assert_launch, bits, fill_sentinel, guarded, ln_modulate_reference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from tpdm_b200 import _lib

    _lib.load()
    return _lib


def _x(batch, rows, D, g):
    """ordinary rows (std 3, mean 1) with every third row replaced by one of mean ~1e3 and std ~1"""
    x = torch.randn(batch, rows, D, device="cuda", generator=g) * 3 + 1
    x[:, 1::3] = 1e3 + torch.randn(batch, len(range(1, rows, 3)), D, device="cuda", generator=g)
    return x


def _mod(batch, D, g):
    """the adaLN layout: six D-wide chunks per batch entry (mod_stride = 6 D)"""
    return torch.randn(batch, 6 * D, device="cuda", generator=g)


@pytest.mark.parametrize("rows", [1, 31, 32, 33, 333])
@pytest.mark.parametrize("D", [1536, 384, 512, 2432])
def test_ln_modulate_routes(L, D, rows):
    """D = 1536 bulk, 384 register kernel <3>, 512 and 2432 (SD3.5-large) the generic <0>; shift and scale read from chunks 3 and 4
    of the 6 D-wide modulation rows."""
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(D + rows)
    for batch in (2, 6):
        x, mod = _x(batch, rows, D, g), _mod(batch, D, g)
        shift, scale = mod[:, 3 * D:4 * D], mod[:, 4 * D:5 * D]
        x0, mod0 = x.clone(), mod.clone()
        buf, out = guarded((batch, rows, D), torch.bfloat16)
        before = buf.clone()
        L.check(lib.tpdm_ln_modulate(L.ptr(x), L.ptr(mod) + 3 * D * 4, L.ptr(mod) + 4 * D * 4, 6 * D, L.ptr(out), batch, rows, D, None))
        torch.cuda.synchronize()
        assert torch.equal(bits(x), bits(x0)) and torch.equal(bits(mod), bits(mod0))
        ref, mag = ln_modulate_reference(x, shift, scale)
        assert_launch(buf, before, [(out, ref, mag, None)], TAU_LN, f"ln_modulate D={D} rows={rows} batch={batch}")


@pytest.mark.parametrize("swap", [False, True])
@pytest.mark.parametrize("N,T,D", [(4096, 333, 1536), (4096, 333, 2432), (1024, 77, 1536)])
def test_ln_modulate_two_segments(L, N, T, D, swap):
    """One launch over image rows (segment 0, N per batch entry) and text rows (segment 1, T): the blocks0 split of the grid,
    each segment's own modulation chunks (swap: the last block's (scale, shift) order of the text stream), and sentinels
    before, between and after the two outputs."""
    lib = L.load()
    batch = 2
    g = torch.Generator(device="cuda").manual_seed(N + T + D + swap)
    x0, x1, mod = _x(batch, N, D, g), _x(batch, T, D, g), _mod(batch, D, g)
    sh1, sc1 = (4, 3) if swap else (3, 4)
    chunk = lambda c: mod[:, c * D:(c + 1) * D]
    at = lambda c: L.ptr(mod) + c * D * 4
    n0, n1, pad = batch * N * D, batch * T * D, 4096
    buf = fill_sentinel(torch.empty(pad + n0 + pad + n1 + pad, dtype=torch.bfloat16, device="cuda"))
    out0 = buf[pad:pad + n0].view(batch, N, D)
    out1 = buf[2 * pad + n0:2 * pad + n0 + n1].view(batch, T, D)
    before = buf.clone()
    inputs = [t.clone() for t in (x0, x1, mod)]
    L.check(lib.tpdm_ln_modulate_pair(L.ptr(x0), at(0), at(1), out0.data_ptr(), N, L.ptr(x1), at(sh1), at(sc1), out1.data_ptr(), T, 6 * D,
                                      batch, D, None))
    torch.cuda.synchronize()
    assert all(torch.equal(bits(a), bits(b)) for a, b in zip((x0, x1, mod), inputs))
    ref0, mag0 = ln_modulate_reference(x0, chunk(0), chunk(1))
    ref1, mag1 = ln_modulate_reference(x1, chunk(sh1), chunk(sc1))
    assert_launch(buf, before, [(out0, ref0, mag0, None), (out1, ref1, mag1, None)], TAU_LN,
                  f"ln_modulate pair N={N} T={T} D={D} swap={swap}")

