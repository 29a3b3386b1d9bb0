"""CPU tests of the element-wise checker the kernel tests use (tests/kernel_check.py) and of the host-side argument checks of
the grouped-GEMM and launch-guard entries: each corruption below must be flagged, and the first two would have passed the
rel-L2 < 6e-3 bar the bf16 GEMM tests used before."""
import ctypes as C

import pytest
import torch

from kernel_check import TAU, assert_close, assert_launch, bits, fill_sentinel, gemm_magnitude

OLD_BF16_REL_TOL = 6e-3


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


@pytest.fixture(scope="module")
def gemm():
    """A bf16 GEMM's float64 reference, its magnitude M and the reference rounded once to bf16 (a perfect kernel's output)."""
    g = torch.Generator().manual_seed(0)
    A = (torch.randn(2, 256, 256, generator=g) * 0.5).bfloat16()
    W = (torch.randn(1024, 256, generator=g) * 0.05).bfloat16()
    bias = torch.randn(1024, generator=g)
    ref = A.double() @ W.double().t() + bias.double()
    return ref, gemm_magnitude(A, W, bias), ref.bfloat16()


def test_clean_bf16_rounded_reference_passes(gemm):
    ref, M, out = gemm
    assert assert_close(out, ref, M, what="clean") <= TAU
    assert assert_close(ref.float(), ref, M, what="clean fp32") <= TAU


def test_one_eight_column_group_four_ulps_off_is_flagged(gemm):
    ref, M, clean = gemm
    out = clean.clone()
    b, r, c = (int(i) for i in torch.unravel_index((ref.abs() / M).argmax(), ref.shape))
    c -= c % 8
    bits(out)[b, r, c:c + 8] += 4          # magnitude + 4 ulps
    assert _rel(out, ref) < OLD_BF16_REL_TOL
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_close(out, ref, M, what="8-column group")


def test_one_32x32_block_scaled_by_1_01_is_flagged(gemm):
    ref, M, clean = gemm
    out = clean.clone()
    out[1, 64:96, 512:544] = (ref[1, 64:96, 512:544] * 1.01).bfloat16()
    assert _rel(out, ref) < OLD_BF16_REL_TOL
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_close(out, ref, M, what="32x32 block")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_one_changed_sentinel_byte_is_flagged(gemm, dtype):
    ref, M, _ = gemm
    buf = fill_sentinel(torch.empty(2, 300, 1024, dtype=dtype))
    assert bool(torch.isnan(buf).all())
    before = buf.clone()
    view = buf[:, 20:276]
    view.copy_(ref.to(dtype))
    writes = [(view, ref, M, None)]
    assert_launch(buf, before, writes, what="clean")
    raw = buf.view(torch.uint8).view(-1)
    k = 276 * 1024 * buf.element_size() + 3   # one byte of the first guard row after batch entry 0's region
    raw[k] ^= 0x01
    with pytest.raises(AssertionError, match="outside the written regions"):
        assert_launch(buf, before, writes, what="changed byte")
    raw[k] ^= 0x01
    view[1, -1, -1] = float("nan")            # an owned element left unwritten (still NaN) fails the element check
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_launch(buf, before, writes, what="unwritten element")


def test_gelu_term_only_widens_by_the_tanh_approximation(gemm):
    ref, M, _ = gemm
    x = ref
    y = torch.nn.functional.gelu(x, approximate="tanh")
    t = torch.tanh(0.7978845608028654 * (x + 0.044715 * x ** 3))
    approx = 0.5 * x * (1 + t + 2.0 ** -11 * torch.sign(x))         # tanh off by 2^-11, the size of tanh.approx.f32's error
    assert assert_close(approx.float(), y, M, gelu_x=x, what="gelu") <= TAU
    with pytest.raises(AssertionError):
        assert_close((0.5 * x * (1 + t + 2.0 ** -6)).float(), y, M, gelu_x=x, what="gelu 2^-6")


# ---------------------------------------------------------------------------------------------------------------
# the C entries: struct layout and the argument errors raised before any CUDA call
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from tpdm_b200 import build
    from tpdm_b200 import _lib as L

    build.build()
    return L.load()


def test_gemm_op_desc_layout():
    from tpdm_b200 import _lib as L

    D = L.TpdmGemmOpDesc
    assert C.sizeof(D) == 10 * 8 + 8 * 4
    assert D.a_row_stride.offset == 8 and D.W.offset == 24 and D.w_scale.offset == 72
    assert D.rows.offset == 80 and D.ksplit.offset == 108


def _desc(**kw):
    from tpdm_b200 import _lib as L

    # pointers that are never dereferenced: every descriptor below fails its argument check first
    d = L.TpdmGemmOpDesc(A=0x1000, W=0x2000, out=0x3000, a_row_stride=64, a_batch_stride=64 * 128, out_batch_stride=256 * 128, rows=128,
                         batch=1, K=64, N=256, epi=0, ldo=256, gate_stride=256, ksplit=1)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _gemm_ops(lib, descs, n=None):
    from tpdm_b200 import _lib as L

    arr = (L.TpdmGemmOpDesc * max(1, len(descs)))(*descs)
    L.check(lib.tpdm_gemm_ops(arr, len(descs) if n is None else n, None))


@pytest.mark.parametrize("case", ["n_ops=0", "n_ops=3", "null ops", "epi 4", "epi -1", "a_scale only", "w_scale only", "null A",
                                  "null W", "null out", "second op bad"])
def test_gemm_ops_argument_errors(lib, case):
    from tpdm_b200 import _lib as L

    bad = {"epi 4": dict(epi=4), "epi -1": dict(epi=-1), "a_scale only": dict(a_scale=0x4000), "w_scale only": dict(w_scale=0x4000),
           "null A": dict(A=None), "null W": dict(W=None), "null out": dict(out=None)}
    with pytest.raises(ValueError):
        if case == "n_ops=0":
            _gemm_ops(lib, [_desc(epi=4)], n=0)
        elif case == "n_ops=3":
            _gemm_ops(lib, [_desc(epi=4)] * 3)
        elif case == "null ops":
            L.check(lib.tpdm_gemm_ops(None, 1, None))
        elif case == "second op bad":
            _gemm_ops(lib, [_desc(), _desc(a_scale=0x4000)])
        else:
            _gemm_ops(lib, [_desc(**bad[case])])
    assert b"tpdm_gemm_ops" in lib.tpdm_last_error()


def test_set_launch_guards_argument_errors(lib):
    from tpdm_b200 import _lib as L

    for slots in (0, -1):
        with pytest.raises(ValueError, match="slots"):
            L.check(lib.tpdm_set_launch_guards(None, None, slots))
    L.check(lib.tpdm_set_launch_guards(None, None, 1))
