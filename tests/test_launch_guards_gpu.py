"""Grouped GEMM launches in the MMDiT's own layouts, the two launch guards of the device-side prompt queue (skip flag and batch
mask) and split K, each against a float64 reference element by element (tests/kernel_check.py) with every byte outside the
launch's own regions checked against the sentinel or the prior residual (run with -m gpu on a B200)."""
import contextlib

import pytest
import torch

from kernel_check import assert_close, assert_launch, bits, gemm_magnitude, guarded

pytestmark = pytest.mark.gpu

DEV = "cuda"
BK = 64   # k-block of the 1-CTA kernel: split K cuts K into ranges of whole k-blocks


@pytest.fixture(scope="module")
def L():
    from tpdm_b200 import _lib

    lib = _lib.load()
    yield _lib
    lib.tpdm_set_launch_guards(None, None, 1)


@contextlib.contextmanager
def guards(L, skip=None, mask=None, slots=1):
    lib = L.load()
    L.check(lib.tpdm_set_launch_guards(L.ptr(skip), L.ptr(mask), slots))
    try:
        yield
    finally:
        L.check(lib.tpdm_set_launch_guards(None, None, 1))


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(g, *shape, scale=1.0):
    return torch.randn(*shape, device=DEV, generator=g) * scale


def _desc(L, A, W, out, rows, batch, K, N, epi, *, a_batch_stride, out_batch_stride, ldo, a_row_stride=None, bias=None, gate=None,
          gate_stride=0, a_scale=None, w_scale=None, ksplit=1):
    """A / out may be tensor views (their data_ptr is used); strides in elements"""
    p = lambda t: None if t is None else t.data_ptr()
    return L.TpdmGemmOpDesc(A=p(A), a_row_stride=K if a_row_stride is None else a_row_stride, a_batch_stride=a_batch_stride, W=p(W),
                            out=p(out), out_batch_stride=out_batch_stride, bias=p(bias), gate=p(gate), a_scale=p(a_scale),
                            w_scale=p(w_scale), rows=rows, batch=batch, K=K, N=N, epi=epi, ldo=ldo, gate_stride=gate_stride, ksplit=ksplit)


def _gemm_ops(L, descs):
    arr = (L.TpdmGemmOpDesc * len(descs))(*descs)
    L.check(L.load().tpdm_gemm_ops(arr, len(descs), None))


def _quantize(L, x):
    x = x.float().contiguous()
    codes = torch.empty(x.shape, dtype=torch.uint8, device=DEV)
    scales = torch.empty(x.shape[:-1], dtype=torch.float32, device=DEV)
    L.check(L.load().tpdm_quantize_fp8_rows(L.ptr(x), x.numel() // x.shape[-1], x.shape[-1], L.ptr(codes), L.ptr(scales), None))
    return codes, scales


def _deq(codes, scales):
    return codes.view(torch.float8_e4m3fn).double() * scales.double().unsqueeze(-1)


class Launch:
    """One launch on fixed inputs.  outs: (buf, view) per output -- view [Bt, ...] inside the guarded allocation buf; `before`
    holds what each buf is reset to before every launch (sentinels, and the prior residual of epi 3).  expect() gives, per
    output, the regions the launch owns with their float64 reference (kernel_check.assert_launch).  `inputs` keeps every tensor
    the launch reads by raw pointer alive for as long as the Launch is."""

    def __init__(self, run, outs, expect=None, inputs=()):
        self.run, self.outs, self.expect, self.inputs = run, outs, expect, inputs
        self.before = [buf.clone() for buf, _ in outs]

    def launch(self, L, skip=None, mask=None, slots=1):
        for (buf, _), b in zip(self.outs, self.before):
            buf.copy_(b)
        with guards(L, skip, mask, slots):
            self.run()
        torch.cuda.synchronize()
        return [buf.clone() for buf, _ in self.outs]

    def check(self, what):
        return max(assert_launch(buf, before, writes, what=what) for (buf, _), before, writes in zip(self.outs, self.before, self.expect()))


# ---------------------------------------------------------------------------------------------------------------
# the MMDiT's grouped layouts on the CTA-pair kernel
# ---------------------------------------------------------------------------------------------------------------
def qkv_launch(L, Bt, N, T, cols, ldo, epi, fp8, K=1536, seed=0):
    """QKV form: op 0 = image rows, op 1 = text rows of ONE [Bt][S][ldo] buffer (op 1's out at row N, out_batch_stride S * ldo);
    separate weights and biases per stream, E4M3 with its own row scales per op."""
    g = _gen(seed)
    S = N + T
    acts = [_randn(g, Bt, r, K) for r in (N, T)]
    wf = [_randn(g, cols, K, scale=0.03) for _ in range(2)]
    bias = [_randn(g, cols, scale=0.1) for _ in range(2)]
    if fp8:
        qa, qw = [_quantize(L, a) for a in acts], [_quantize(L, w) for w in wf]
        A, W = [c for c, _ in qa], [c for c, _ in qw]
        a_s, w_s = [s for _, s in qa], [s for _, s in qw]
        A64, W64 = [_deq(*q) for q in qa], [_deq(*q) for q in qw]
    else:
        A, W = [(a * 0.5).bfloat16() for a in acts], [w.bfloat16() for w in wf]
        a_s = w_s = [None, None]
        A64, W64 = [a.double() for a in A], [w.double() for w in W]
    buf, out = guarded((Bt, S, ldo), torch.float32 if epi == 1 else torch.bfloat16)
    descs = [_desc(L, A[i], W[i], out[:, r0:], rows, Bt, K, cols, epi, a_batch_stride=rows * K, out_batch_stride=S * ldo, ldo=ldo,
                   bias=bias[i], a_scale=a_s[i], w_scale=w_s[i]) for i, (r0, rows) in enumerate(((0, N), (N, T)))]

    def expect():
        writes = []
        for i, (r0, r1) in enumerate(((0, N), (N, S))):
            pre = A64[i] @ W64[i].t() + bias[i].double()
            mag = A64[i].abs() @ W64[i].abs().t() + bias[i].double().abs()
            ref = torch.nn.functional.gelu(pre, approximate="tanh") if epi == 2 else pre
            writes.append((out[:, r0:r1, :cols], ref, mag, pre if epi == 2 else None))
        return [writes]

    return Launch(lambda: _gemm_ops(L, descs), [(buf, out)], expect, inputs=(A, W, a_s, w_s, bias))


def outproj_launch(L, Bt, N, T, cols, K, seed=1):
    """Out-projection / FF2 form (epi 3): A strided out of one shared [Bt][S][K] buffer (op 1 starts at row N); outputs are the
    separate image and text residuals, each inside a guarded allocation; gates from a modulation-like [Bt][12 * cols] buffer
    (gate_stride != N) at a different column offset per op."""
    g = _gen(seed)
    S = N + T
    A = _randn(g, Bt, S, K, scale=0.5).bfloat16()
    W = [_randn(g, cols, K, scale=0.05 * (1536 / K) ** 0.5).bfloat16() for _ in range(2)]
    bias = [_randn(g, cols, scale=0.1) for _ in range(2)]
    mod = _randn(g, Bt, 12 * cols)
    gates = [mod[:, 2 * cols:3 * cols], mod[:, 11 * cols:]]
    res = [guarded((Bt, r, cols), torch.float32) for r in (N, T)]
    for _, v in res:
        v.copy_(_randn(g, *v.shape))
    descs = [_desc(L, A[:, r0:], W[i], res[i][1], rows, Bt, K, cols, 3, a_batch_stride=S * K, out_batch_stride=rows * cols, ldo=cols,
                   bias=bias[i], gate=gates[i], gate_stride=12 * cols) for i, (r0, rows) in enumerate(((0, N), (N, T)))]
    launch = Launch(lambda: _gemm_ops(L, descs), res, inputs=(A, W, bias, mod))
    prior = [v.double() for _, v in res]

    def expect():
        writes = []
        for i, (r0, r1) in enumerate(((0, N), (N, S))):
            a, gt = A[:, r0:r1].double(), gates[i].double()[:, None, :]
            pre = a @ W[i].double().t() + bias[i].double()
            mag = gt.abs() * (a.abs() @ W[i].double().abs().t() + bias[i].double().abs()) + prior[i].abs()
            writes.append([(res[i][1], prior[i] + gt * pre, mag, None)])
        return writes

    launch.expect = expect
    return launch


QKV_CASES = [(2, 1024, 154, 4608, 4608), (2, 4096, 333, 4608, 4608),
             (6, 333, 77, 392, 392),      # ragged M tiles, a ragged 256-wide N tile, text pairs whose second CTA has no valid row
             (6, 333, 77, 392, 456)]      # ldo = cols + 64: the 64 columns past N stay sentinel


@pytest.mark.parametrize("fp8", [False, True], ids=["bf16", "e4m3"])
@pytest.mark.parametrize("epi", [0, 1, 2])
@pytest.mark.parametrize("Bt,N,T,cols,ldo", QKV_CASES)
def test_grouped_qkv_layout(L, Bt, N, T, cols, ldo, epi, fp8):
    c = qkv_launch(L, Bt, N, T, cols, ldo, epi, fp8)
    c.launch(L)
    c.check(f"qkv {'e4m3' if fp8 else 'bf16'} Bt={Bt} N={N} T={T} cols={cols} ldo={ldo} epi={epi}")


@pytest.mark.parametrize("Bt,N,T,cols,K", [(2, 1024, 154, 1536, 1536), (2, 1024, 154, 1536, 6144), (6, 333, 77, 392, 1536)])
def test_grouped_outproj_ff2_layout(L, Bt, N, T, cols, K):
    c = outproj_launch(L, Bt, N, T, cols, K)
    c.launch(L)
    c.check(f"out-proj Bt={Bt} N={N} T={T} cols={cols} K={K}")


# ---------------------------------------------------------------------------------------------------------------
# skip flag and batch mask, every guarded kernel family
# ---------------------------------------------------------------------------------------------------------------
def proj_out_launch(L, Bt, rows=1024, N=64, K=1536, seed=2):
    """the 1-CTA kernel at proj_out's shape (N = 64, fp32 out) through tpdm_gemm_bf16"""
    g = _gen(seed)
    A, W, bias = _randn(g, Bt, rows, K, scale=0.5).bfloat16(), _randn(g, N, K, scale=0.05).bfloat16(), _randn(g, N)
    buf, out = guarded((Bt, rows, N), torch.float32)
    lib = L.load()
    return Launch(lambda: L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), None, L.ptr(out), Bt, rows, N, K, 1, None)),
                  [(buf, out)])


def conv1_launch(L, Bt, g_side=64, C=3072, N=128, seed=3):
    """the 1-CTA kernel in implicit-GEMM conv mode at the TimePredictor's conv1 shape"""
    g = _gen(seed)
    x = _randn(g, Bt, g_side, g_side, C).bfloat16()
    w, bias = _randn(g, N, 9 * C, scale=0.02).bfloat16(), _randn(g, N)
    buf, out = guarded((Bt, g_side * g_side, N), torch.float32)
    lib = L.load()
    return Launch(lambda: L.check(lib.tpdm_conv3x3_nhwc(L.ptr(x), L.ptr(w), L.ptr(bias), L.ptr(out), Bt, g_side, C, N, None)),
                  [(buf, out)])


def attention_launch(L, Bt, S, d, H=2, seed=4):
    g = _gen(seed)
    dp = 64 if d <= 64 else 128
    qkv = torch.zeros(Bt, S, 3, H, dp, device=DEV)
    qkv[..., :d] = _randn(g, Bt, S, 3, H, d)
    qkv = qkv.bfloat16()
    buf, out = guarded((Bt, S, H * dp), torch.bfloat16)
    lib = L.load()
    return Launch(lambda: L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, dp, d, 0, None)), [(buf, out)])


def ln_launch(L, Bt, D, fp8, rows=333, seed=5):
    g = _gen(seed)
    x = _randn(g, Bt, rows, D, scale=3.0) + 1
    mod = _randn(g, Bt, 4 * D)
    shift, scale = mod.data_ptr(), mod.data_ptr() + 4 * D    # bytes: scale = columns [D, 2D)
    lib = L.load()
    if fp8:
        cb, codes = guarded((Bt, rows, D), torch.uint8)
        sb, scales = guarded((Bt, rows), torch.float32)
        return Launch(lambda: L.check(lib.tpdm_ln_modulate_fp8(L.ptr(x), shift, scale, 4 * D, L.ptr(codes), L.ptr(scales), Bt, rows, D, None)),
                      [(cb, codes), (sb, scales)], inputs=(x, mod))
    buf, out = guarded((Bt, rows, D), torch.bfloat16)
    return Launch(lambda: L.check(lib.tpdm_ln_modulate(L.ptr(x), shift, scale, 4 * D, L.ptr(out), Bt, rows, D, None)), [(buf, out)],
                  inputs=(x, mod))


FAMILIES = {
    "gemm2_bf16_epi0": lambda L, Bt: qkv_launch(L, Bt, 333, 77, 392, 392, 0, False),
    "gemm2_bf16_epi3": lambda L, Bt: outproj_launch(L, Bt, 333, 77, 392, 1536),
    "gemm2_e4m3": lambda L, Bt: qkv_launch(L, Bt, 333, 77, 392, 392, 0, True),
    "gemm1_proj_out": proj_out_launch,
    "gemm1_conv1": conv1_launch,
    "attention_s4429_d64": lambda L, Bt: attention_launch(L, Bt, 4429, 64),
    "attention_s589_d96": lambda L, Bt: attention_launch(L, Bt, 589, 96, H=3),
    "ln_modulate_d1536": lambda L, Bt: ln_launch(L, Bt, 1536, False),
    "ln_modulate_d384": lambda L, Bt: ln_launch(L, Bt, 384, False),
    "ln_modulate_fp8_d1536": lambda L, Bt: ln_launch(L, Bt, 1536, True),
}


def _per_batch(t, view):
    """the [Bt, ...] view `view` has inside its allocation, applied to a copy t of that allocation"""
    return t.as_strided(view.shape, view.stride(), view.storage_offset())


def _assert_bits_equal(got, expected, outs, what):
    for k, (gt, ex, (_, view)) in enumerate(zip(got, expected, outs)):
        if not torch.equal(bits(gt), bits(ex)):
            pg, pe = _per_batch(bits(gt), view), _per_batch(bits(ex), view)
            rows = [b for b in range(view.shape[0]) if not torch.equal(pg[b], pe[b])]
            raise AssertionError(f"{what}: output {k} differs in batch entries {rows}" + ("" if rows else " (outside the output view)"))


def _patterns(slots):
    return {"all on": [1] * slots, "all off": [0] * slots, "one on": [int(s == 1) for s in range(slots)],
            "alternating": [int(s % 2 == 0) for s in range(slots)]}


@pytest.mark.parametrize("slots", [2, 3, 4])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_batch_mask(L, family, slots):
    """Bt = 2 * slots (the CFG halves b and b + slots share a slot): entries of active slots are bit-identical to an unguarded
    launch, entries of masked slots keep their prior contents bit for bit."""
    Bt = 2 * slots
    c = FAMILIES[family](L, Bt)
    plain = c.launch(L)
    assert not all(torch.equal(bits(p), bits(b)) for p, b in zip(plain, c.before)), "the unguarded launch wrote nothing"
    for name, pattern in _patterns(slots).items():
        mask = torch.tensor(pattern, dtype=torch.int32, device=DEV)
        got = c.launch(L, mask=mask, slots=slots)
        expected = [b.clone() for b in c.before]
        for ex, p, (_, view) in zip(expected, plain, c.outs):
            for b in range(Bt):
                if pattern[b % slots]:
                    _per_batch(ex, view)[b] = _per_batch(p, view)[b]
        _assert_bits_equal(got, expected, c.outs, f"{family} slots={slots} mask {name} {pattern}")


@pytest.mark.parametrize("family", list(FAMILIES))
def test_skip_flag(L, family):
    """A device flag of 1 leaves every output untouched; 0 gives the unguarded result bit for bit, and so does a launch after
    the guards were cleared."""
    lib = L.load()
    c = FAMILIES[family](L, 4)
    plain = c.launch(L)
    one, zero = torch.ones(1, dtype=torch.int32, device=DEV), torch.zeros(1, dtype=torch.int32, device=DEV)
    _assert_bits_equal(c.launch(L, skip=one), c.before, c.outs, f"{family} skip flag 1")
    _assert_bits_equal(c.launch(L, skip=zero), plain, c.outs, f"{family} skip flag 0")
    L.check(lib.tpdm_set_launch_guards(L.ptr(one), L.ptr(torch.zeros(4, dtype=torch.int32, device=DEV)), 4))
    L.check(lib.tpdm_set_launch_guards(None, None, 1))
    for (buf, _), b in zip(c.outs, c.before):
        buf.copy_(b)
    c.run()
    torch.cuda.synchronize()
    _assert_bits_equal([buf for buf, _ in c.outs], plain, c.outs, f"{family} after clearing the guards")


# ---------------------------------------------------------------------------------------------------------------
# split K on the 1-CTA kernel (the decode_tile / K-range code TimePredictor.conv1 runs with ksplit = 4)
# ---------------------------------------------------------------------------------------------------------------
SPLIT_K = [   # (batch, rows, N, K, ksplit, mask over 2 slots or None)
    (1, 200, 128, 1000, 3, None),      # 16 k-blocks, the last one 40 elements: ranges of 6 / 6 / 4
    (1, 200, 64, 1000, 16, None),      # one k-block per range
    (2, 300, 128, 1000, 3, None),
    (4, 130, 128, 1000, 3, [1, 0]),    # entries 1 and 3 masked
]


@pytest.mark.parametrize("batch,rows,N,K,ksplit,pattern", SPLIT_K)
def test_split_k(L, batch, rows, N, K, ksplit, pattern):
    g = _gen(6)
    A, W = _randn(g, batch, rows, K, scale=0.5).bfloat16(), _randn(g, N, K, scale=0.05).bfloat16()
    buf, out = guarded((ksplit, batch, rows, N), torch.float32)
    before = buf.clone()
    d = _desc(L, A, W, out, rows, batch, K, N, 1, a_batch_stride=rows * K, out_batch_stride=rows * N, ldo=N, ksplit=ksplit)
    mask = None if pattern is None else torch.tensor(pattern, dtype=torch.int32, device=DEV)
    with guards(L, mask=mask, slots=len(pattern) if pattern else 1):
        _gemm_ops(L, [d])
    torch.cuda.synchronize()
    nkb = (K + BK - 1) // BK
    kps = (nkb + ksplit - 1) // ksplit
    ranges = [(s * kps, min((s + 1) * kps, nkb)) for s in range(ksplit)]
    if (K, ksplit) == (1000, 3):
        assert [e - b for b, e in ranges] == [6, 6, 4]
    active = [b for b in range(batch) if pattern is None or pattern[b % len(pattern)]]
    A64, W64 = A.double(), W.double()
    writes = []
    for s, (kb0, kb1) in enumerate(ranges):
        k0, k1 = kb0 * BK, min(kb1 * BK, K)
        for b in active:
            writes.append((out[s, b], A64[b, :, k0:k1] @ W64[:, k0:k1].t(), gemm_magnitude(A[b, :, k0:k1], W[:, k0:k1]), None))
    assert_launch(buf, before, writes, what=f"split K {batch}x{rows}x{N}x{K} ksplit {ksplit} mask {pattern}")
    total = out[:, active].double().sum(0)
    assert_close(total, A64[active] @ W64.t(), gemm_magnitude(A[active], W), what="sum of the split-K slabs")


def test_split_k_rejects_unsupported_ops(L):
    g = _gen(7)
    A = _randn(g, 1, 128, 1000).bfloat16()
    W, W256 = _randn(g, 128, 1000).bfloat16(), _randn(g, 256, 1000).bfloat16()
    A320, W320 = A[..., :320].contiguous(), W[:, :320].contiguous()     # 5 k-blocks: ranges of 2 leave the 4th empty
    bias = _randn(g, 256)
    out = torch.zeros(4, 128, 256, device=DEV)
    kw = dict(out_batch_stride=128 * 256, ldo=256)
    cases = {"bias": _desc(L, A, W, out, 128, 1, 1000, 128, 1, bias=bias, ksplit=2, a_batch_stride=128 * 1000, **kw),
             "bf16 output": _desc(L, A, W, out, 128, 1, 1000, 128, 0, ksplit=2, a_batch_stride=128 * 1000, **kw),
             "N > 128": _desc(L, A, W256, out, 128, 1, 1000, 256, 1, ksplit=2, a_batch_stride=128 * 1000, **kw),
             "empty range": _desc(L, A320, W320, out, 128, 1, 320, 128, 1, ksplit=4, a_batch_stride=128 * 320, **kw)}
    before = out.clone()
    for name, d in cases.items():
        with pytest.raises(ValueError):
            _gemm_ops(L, [d])
    torch.cuda.synchronize()
    assert torch.equal(out, before)
