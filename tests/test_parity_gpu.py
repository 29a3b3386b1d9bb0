"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C-ABI against the fp32 oracle and the golden
fixtures.  Tolerances are BASELINE.json's: per-step velocity <= 2e-2 rel-L2, sigma sequence <= 1e-3 abs, final latent
<= 3e-2 rel-L2 (bf16 tensor-core path vs fp32 oracle)."""
import math

import pytest
import torch

from kernel_check import assert_launch, gemm_magnitude, guarded

pytestmark = pytest.mark.gpu

VEL_TOL, SIGMA_TOL, LATENT_TOL = 2e-2, 1e-3, 3e-2


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def L():
    from tpdm_b200 import _lib

    _lib.load()
    return _lib


# ---------------------------------------------------------------------------------------------------------------
# unit kernels through the C-ABI
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch,rows,N,K,epi", [
    (1, 128, 256, 64, 1), (2, 333, 384, 384, 0), (2, 333, 1152, 384, 2), (2, 256, 384, 1536, 3), (2, 256, 64, 384, 1),
    (1, 1, 8, 64, 1), (3, 130, 200, 72, 0), (2, 1024, 4608, 1536, 0), (2, 1024, 1536, 6144, 3)])
def test_gemm(L, batch, rows, N, K, epi):
    """every element against the float64 reference (tests/kernel_check.py); nothing written outside [batch][rows][N]"""
    torch.manual_seed(0)
    lib = L.load()
    dev = "cuda"
    A = (torch.randn(batch, rows, K, device=dev) * 0.5).bfloat16()
    W = (torch.randn(N, K, device=dev) * 0.05).bfloat16()
    bias, gate = torch.randn(N, device=dev), torch.randn(batch, N, device=dev)
    pre = A.double() @ W.double().t() + bias.double()
    mag = gemm_magnitude(A, W, bias)
    buf, out = guarded((batch, rows, N), torch.bfloat16 if epi in (0, 2) else torch.float32)
    ref = torch.nn.functional.gelu(pre, approximate="tanh") if epi == 2 else pre
    if epi == 3:
        out.copy_(torch.randn(batch, rows, N, device=dev))
        g = gate.double()[:, None, :]
        ref, mag = out.double() + g * pre, g.abs() * mag + out.double().abs()
    before = buf.clone()
    L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), L.ptr(gate), L.ptr(out), batch, rows, N, K, epi, None))
    torch.cuda.synchronize()
    assert_launch(buf, before, [(out, ref, mag, pre if epi == 2 else None)], what=f"gemm {batch}x{rows}x{N}x{K} epi {epi}")


def test_gemm_rejects_bad_arguments(L):
    lib = L.load()
    A = torch.zeros(1, 8, 60, device="cuda", dtype=torch.bfloat16)
    W = torch.zeros(8, 60, device="cuda", dtype=torch.bfloat16)
    out = torch.zeros(1, 8, 8, device="cuda")
    with pytest.raises(ValueError):
        L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), None, None, L.ptr(out), 1, 8, 8, 60, 1, None))   # K % 8 != 0
    with pytest.raises(ValueError):
        L.check(lib.tpdm_gemm_bf16(None, L.ptr(W), None, None, L.ptr(out), 1, 8, 8, 64, 1, None))
    with pytest.raises(ValueError):
        L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), None, None, L.ptr(out), 1, 8, 8, 64, 3, None))   # gate missing


@pytest.mark.parametrize("Bt,S,H,d,q_rows", [(1, 128, 1, 64, 0), (1, 1, 1, 64, 0), (2, 589, 4, 96, 0), (1, 1357, 4, 64, 0),
                                             (1, 1357, 4, 64, 1024), (2, 300, 3, 32, 0), (1, 4429, 2, 64, 0)])
def test_joint_attention(L, Bt, S, H, d, q_rows):
    torch.manual_seed(1)
    lib = L.load()
    dp = 64 if d <= 64 else 128
    qkv = torch.zeros(Bt, S, 3, H, dp, device="cuda")
    qkv[..., :d] = torch.randn(Bt, S, 3, H, d, device="cuda") * 1.5
    qkv = qkv.bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, dp, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i, :, :d].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2)
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, dp, d, q_rows, None))
    torch.cuda.synchronize()
    rows = q_rows or S
    assert rel(out[:, :rows, :, :d], ref[:, :rows]) < 6e-3
    if dp > d:
        assert float(out[..., d:].float().abs().max()) == 0.0
    # ordinary activations never leave the fast kernel (the exact kernel behind it is an empty launch)
    assert lib.tpdm_attention_redo_count() in (0, -1)


@pytest.mark.parametrize("jump", [10, 40, 70, 100, 300, 330, 370, 511, "ramp"])
def test_attention_large_logits_trigger_rescale(L, jump):
    """Rows whose running max grows by far more than 2^32 between keys exercise the lazy reference update: the jump is placed
    in every 32-key chunk position of a 128-key tile (chunks 0/1 are rescaled before their P is handed to the MMA warp, chunks
    2/3 after the first half of P V has been issued), in the first and in later tiles, and as a ramp that moves it many times."""
    torch.manual_seed(2)
    lib = L.load()
    Bt, S, H, d = 1, 512, 2, 64
    qkv = torch.randn(Bt, S, 3, H, d, device="cuda")
    qkv[:, :, 0] *= 6.0
    if jump == "ramp":
        qkv[:, :, 1] *= torch.linspace(0.5, 12.0, S, device="cuda").view(1, S, 1, 1)
    else:
        qkv[:, jump:, 1] *= 6.0     # later keys carry much larger logits
    qkv = qkv.bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2)
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, 64, d, 0, None))
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    assert rel(out, ref) < 1e-2


def test_attention_extreme_logits_stay_finite(L):
    """Scores of +-1e4 (far beyond exp range in fp32 without a reference): softmax degenerates to a one-hot pick of the arg-max key."""
    torch.manual_seed(9)
    lib = L.load()
    Bt, S, H, d = 1, 384, 1, 64
    qkv = torch.randn(Bt, S, 3, H, d, device="cuda")
    qkv[:, :, 0] *= 40.0
    qkv[:, :, 1] *= 40.0
    qkv = qkv.bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2)
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, 64, d, 0, None))
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    assert rel(out, ref) < 1e-2
    # scores this far apart cannot be kept in range by the row-sum guard of the fast kernel: its CTAs must have been flagged and
    # recomputed by the exact kernel (per-chunk maxima)
    n_redo = lib.tpdm_attention_redo_count()
    assert n_redo == -1 or n_redo > 0, n_redo


@pytest.mark.parametrize("scale_k", [2.0, 3.0, 4.5])
def test_attention_row_sum_guard_moves_the_reference(L, scale_k):
    """Keys whose scores grow steadily (a few 2^10 per 128-key tile) are handled INSIDE the fast kernel: the row sum crosses 2^32
    at the top of a tile and the reference is moved by floor(log2 l) (O and l rescaled) -- no tile is handed to the exact kernel."""
    torch.manual_seed(5)
    lib = L.load()
    Bt, S, H, d = 1, 1024, 2, 64
    qkv = torch.randn(Bt, S, 3, H, d, device="cuda")
    qkv[:, :, 0] = qkv[:, :, 0].abs() * 2.0                     # q >= 0 ...
    qkv[:, :, 1] = qkv[:, :, 1].abs() * torch.linspace(0.05, scale_k, S, device="cuda").view(1, S, 1, 1)   # ... k >= 0 and growing
    qkv = qkv.bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2)
    spread = (q @ k.transpose(-1, -2) * (1.4427 / 8)).amax(-1) - (q @ k[:, :, :128].transpose(-1, -2) * (1.4427 / 8)).amax(-1)
    assert float(spread.max()) > 40.0       # log2 units above the first tile's maximum: the guard has to act
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, 64, d, 0, None))
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    assert rel(out, ref) < 1e-2
    n_redo = lib.tpdm_attention_redo_count()
    if scale_k <= 2.0:   # the guard of the eight-softmax-warp build acts every 4th tile; faster growth takes the exact pass (still exact)
        assert n_redo in (0, -1), n_redo


@pytest.mark.parametrize("d", [64, 96])
def test_attention_exact_pass_only_where_needed(L, d):
    """One head carries scores of +-1e4, the others are ordinary: only that head's query tiles may take the exact pass of the fast
    kernel (also in the 128-wide padded-head instantiation, d = 96), and every head must match the fp32 reference."""
    torch.manual_seed(13)
    lib = L.load()
    Bt, S, H = 2, 700, 3
    dp = 64 if d <= 64 else 128
    qkv = torch.zeros(Bt, S, 3, H, dp, device="cuda")
    qkv[..., :d] = torch.randn(Bt, S, 3, H, d, device="cuda")
    qkv[:, :, 0, 1, :d] *= 40.0
    qkv[:, :, 1, 1, :d] *= 40.0
    qkv = qkv.bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, dp, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i, :, :d].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2)
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, dp, d, 0, None))
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    for h in range(H):
        assert rel(out[:, :, h, :d], ref[:, :, h]) < 1e-2, h
    n_redo = lib.tpdm_attention_redo_count()
    q_tiles = (S + 127) // 128
    assert n_redo == -1 or 0 < n_redo <= Bt * q_tiles, n_redo


def test_attention_cold_cache_no_deadlock(L):
    """The fast attention path lets the softmax warps run up to two tiles ahead of the P V issuer.  With K / V tiles coming from HBM
    (L2 flushed) and a copy stream competing for bandwidth, a V tile can arrive thousands of cycles late: the hand-over barriers
    must survive that (an earlier build with single, phase-j&1 barriers dead-locked in the first full denoising step).  Run under
    `timeout` on the GPU box: a regression shows as a hang."""
    torch.manual_seed(11)
    lib = L.load()
    Bt, S, H, d = 2, 4429, 24, 64
    qkv = torch.randn(Bt, S, 3, H, d, device="cuda").bfloat16().contiguous()
    out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
    q, k, v = (qkv[:, :, i].float().transpose(1, 2) for i in range(3))
    ref = torch.nn.functional.scaled_dot_product_attention(q[:1, :4], k[:1, :4], v[:1, :4]).transpose(1, 2)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    big_a = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    big_b = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    first = None
    for it in range(12):
        flush.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for _ in range(3):
                big_b.copy_(big_a)
        L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, 64, d, 0, None))
        torch.cuda.synchronize()
        if first is None:
            first = out.clone()
        else:
            assert torch.equal(out, first)
    assert rel(out[:1, :, :4], ref) < 6e-3
    assert lib.tpdm_attention_redo_count() in (0, -1)


def test_tcgen05_kernels_are_bit_reproducible(L):
    """compute-sanitizer is closed on the GPU pool (profiles/r02_sanitizer_closed.txt), so the hand-rolled mbarrier / TMEM protocols
    are checked the other way a race shows: every kernel must return BIT-identical results when it is run again and again on the
    same inputs (tail tiles, forced reference raises, grouped launches, every epilogue)."""
    torch.manual_seed(17)
    lib = L.load()
    dev = "cuda"
    reps = 12
    for (Bt, S, H, d, big) in ((2, 4429, 6, 64, False), (1, 1357, 4, 64, True), (2, 589, 4, 96, False), (1, 130, 2, 64, True)):
        dp = 64 if d <= 64 else 128
        qkv = torch.zeros(Bt, S, 3, H, dp, device=dev)
        qkv[..., :d] = torch.randn(Bt, S, 3, H, d, device=dev)
        if big:
            qkv[:, :, 0] *= 6.0
            qkv[:, S // 2:, 1] *= 6.0        # the reference maximum is raised half way through
        qkv = qkv.bfloat16().contiguous()
        outs = []
        for _ in range(reps):
            out = torch.zeros(Bt, S, H, dp, device=dev, dtype=torch.bfloat16)
            L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, dp, d, 0, None))
            outs.append(out)
        torch.cuda.synchronize()
        assert all(torch.equal(outs[0], o) for o in outs[1:]), ("attention", Bt, S, H, d)
    for (batch, rows, N, K, epi) in ((2, 4429, 1536, 1536, 3), (2, 4096, 4608, 1536, 0), (2, 333, 6144, 1536, 2), (3, 130, 200, 72, 1), (2, 1024, 64, 1536, 1)):
        A = (torch.randn(batch, rows, K, device=dev) * 0.5).bfloat16()
        W = (torch.randn(N, K, device=dev) * 0.05).bfloat16()
        bias, gate = torch.randn(N, device=dev), torch.randn(batch, N, device=dev)
        base = torch.randn(batch, rows, N, device=dev)
        outs = []
        for _ in range(reps):
            out = base.clone() if epi in (1, 3) else torch.zeros(batch, rows, N, device=dev, dtype=torch.bfloat16)
            L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), L.ptr(gate), L.ptr(out), batch, rows, N, K, epi, None))
            outs.append(out)
        torch.cuda.synchronize()
        assert all(torch.equal(outs[0], o) for o in outs[1:]), ("gemm", batch, rows, N, K, epi)
    x = torch.randn(1, 64, 64, 3072, device=dev).bfloat16()
    w = (torch.randn(128, 9 * 3072, device=dev) * 0.02).bfloat16()
    outs = []
    for _ in range(reps):
        out = torch.zeros(1, 64 * 64, 128, device=dev)
        L.check(lib.tpdm_conv3x3_nhwc(L.ptr(x), L.ptr(w), None, L.ptr(out), 1, 64, 3072, 128, None))
        outs.append(out)
    torch.cuda.synchronize()
    assert all(torch.equal(outs[0], o) for o in outs[1:]), "conv3x3"


@pytest.mark.parametrize("B,g,C,N", [(2, 16, 128, 128), (1, 64, 3072, 128), (1, 8, 64, 128), (1, 128, 128, 128)])
def test_conv3x3_implicit_gemm(L, B, g, C, N):
    torch.manual_seed(3)
    lib = L.load()
    x = torch.randn(B, C, g, g, device="cuda").bfloat16()
    w = (torch.randn(N, C, 3, 3, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(N, device="cuda")
    nhwc = lambda y: y.permute(0, 2, 3, 1).reshape(B, g * g, N)
    ref = nhwc(torch.nn.functional.conv2d(x.double(), w.double(), bias.double(), padding=1))
    mag = nhwc(torch.nn.functional.conv2d(x.double().abs(), w.double().abs(), bias.double().abs(), padding=1))
    xn = x.permute(0, 2, 3, 1).contiguous()
    wp = w.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous()
    buf, out = guarded((B, g * g, N), torch.float32)
    before = buf.clone()
    L.check(lib.tpdm_conv3x3_nhwc(L.ptr(xn), L.ptr(wp), L.ptr(bias), L.ptr(out), B, g, C, N, None))
    torch.cuda.synchronize()
    assert_launch(buf, before, [(out, ref, mag, None)], what=f"conv3x3 B={B} g={g} C={C} N={N}")


def test_ln_modulate(L):
    torch.manual_seed(4)
    lib = L.load()
    B, rows, D = 2, 333, 1536
    x = torch.randn(B, rows, D, device="cuda") * 3 + 1
    mod = torch.randn(B, 4 * D, device="cuda")
    out = torch.zeros(B, rows, D, device="cuda", dtype=torch.bfloat16)
    L.check(lib.tpdm_ln_modulate(L.ptr(x), mod.data_ptr(), mod.data_ptr() + 4 * D, 4 * D, L.ptr(out), B, rows, D, None))
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (D,), eps=1e-6) * (1 + mod[:, None, D:2 * D]) + mod[:, None, :D]
    assert rel(out, ref) < 4e-3


def test_euler_step_matches_reference_fixture(golden):
    from tpdm_b200.model_utilis import CustomFlowMatchEulerDiscreteScheduler

    fx = golden("pieces_ref")
    sch = CustomFlowMatchEulerDiscreteScheduler()
    prev = sch.custom_step(fx["euler.model_output"].cuda(), fx["euler.sigma_next"].cuda(), fx["euler.sigma"].cuda(),
                           fx["euler.sample"].cuda(), return_dict=False)[0]
    assert torch.allclose(prev.cpu(), fx["euler.prev"], atol=1e-6)   # fp32 fma vs mul+add
    assert sch.custom_step(fx["euler.model_output"].cuda(), fx["euler.sigma_next"].cuda(), fx["euler.sigma"].cuda(),
                           fx["euler.sample"].cuda()).prev_sample.shape == prev.shape


# ---------------------------------------------------------------------------------------------------------------
# TimePredictor against the reference's own outputs
# ---------------------------------------------------------------------------------------------------------------
def test_time_predictor_matches_reference_fixture(golden):
    from tpdm_b200.modeling_sd3_pnt import TimePredictor

    fx = golden("tpm_ref")
    tp = TimePredictor(128, 128).cuda()
    tp.load_state_dict({k: v for k, v in fx.items() if not k.startswith("grad.") and k not in ("x", "temb", "alpha_beta")})
    y = tp(fx["x"].cuda(), fx["temb"].cuda())
    assert y.shape == (2, 2)
    assert torch.allclose(y.cpu(), fx["alpha_beta"], rtol=3e-3), (y.cpu(), fx["alpha_beta"])


def test_time_predictor_sd3m_shape_vs_oracle():
    from oracle import sd3_oracle as O
    from tpdm_b200.modeling_sd3_pnt import TimePredictor

    torch.manual_seed(5)
    ora = O.OracleTimePredictor(128, 3072).cuda()
    with torch.no_grad():   # make the head input-sensitive (the default init is bias dominated)
        ora.fc2.weight.mul_(20)
        ora.fc1.weight.mul_(5)
    tp = TimePredictor(128, 3072).cuda()
    tp.load_state_dict(ora.state_dict())
    x = torch.randn(1, 3072, 64, 64, device="cuda")
    temb = torch.randn(1, 1536, device="cuda")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    with torch.no_grad():
        ref = ora(x, temb)
    got = tp(x, temb)
    assert torch.allclose(got, ref, rtol=5e-3), (got, ref)


# ---------------------------------------------------------------------------------------------------------------
# MMDiT forward and the adaptive loop, tiny config (BASELINE.json configs[0])
# ---------------------------------------------------------------------------------------------------------------
def _tiny(qk_norm=None):
    from oracle import sd3_oracle as O
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    cfg = O.tiny_config(qk_norm=qk_norm)
    pipe = O.build_pipeline(cfg)
    inp = O.synthetic_inputs(cfg, batch=2)
    tcfg = dict(sample_size=32, num_layers=2, attention_head_dim=96, num_attention_heads=4, caption_projection_dim=384,
                pos_embed_max_size=96, qk_norm=qk_norm)
    model = SD3PredictNextTimeStepModel(transformer_config=tcfg, torch_dtype=torch.float32, device="cuda")
    model.transformer.load_state_dict(pipe.transformer.state_dict())
    model.time_predictor.load_state_dict(pipe.time_predictor.state_dict())
    return pipe, inp, model


def test_mmdit_forward_tiny_vs_golden(golden):
    pipe, inp, model = _tiny()
    fx = golden("tiny_block")
    lat2 = torch.cat([inp["latents"]] * 2).cuda()
    pe = torch.cat([inp["negative_prompt_embeds"], inp["prompt_embeds"]]).cuda()
    pp = torch.cat([inp["negative_pooled_prompt_embeds"], inp["pooled_prompt_embeds"]]).cuda()
    v, temb, h1, h2 = model.transformer(lat2, pe, pp, fx["timestep"].cuda(), return_dict=False)
    assert v.shape == (4, 16, 32, 32) and temb.shape == (4, 384) and h1.shape == (4, 256, 384) and h2.shape == (4, 256, 384)
    assert rel(temb, fx["temb"]) < 1e-4
    assert rel(h1[:, 0], fx["h1_row0"]) < 1e-5
    assert rel(h2[:, 17], fx["h2_tok17"]) < VEL_TOL
    assert rel(v, fx["velocity"]) < VEL_TOL
    out = model.transformer(lat2, pe, pp, fx["timestep"].cuda())
    assert torch.equal(out.sample, v) and torch.equal(out["hidden_states_2"], h2)


@pytest.mark.parametrize("qk_norm", [None, "rms_norm"])
def test_tiny_trajectory_vs_golden(golden, qk_norm):
    pipe, inp, model = _tiny(qk_norm)
    fx = golden("tiny_traj" if qk_norm is None else "tiny_traj_qknorm")
    cu = {k: v.cuda() for k, v in inp.items()}
    out = model(**cu, max_inference_steps=8, guidance_scale=7.0, predict=True, return_velocities=True)
    T = fx["sigmas"].shape[1]
    assert out.sigmas.shape == (2, T)
    assert float((out.sigmas.cpu() - fx["sigmas"]).abs().max()) < SIGMA_TOL
    assert torch.equal(out.prob_masks.cpu().to(torch.uint8), fx["prob_masks"])
    assert float((out.alphas.cpu() - fx["alphas"]).abs().max()) < 2e-2
    assert float((out.logprobs.cpu() - fx["logprobs"]).abs().max()) < 5e-3
    for t in range(T):
        assert rel(out["velocities"][:, t], fx["velocities"][:, t]) < VEL_TOL, t
    assert rel(out.latents, fx["final_latents"]) < LATENT_TOL
    assert [int(i) for i in out.last_valid_indices] == fx["last_valid_indices"].tolist()
    assert rel(out.tembs, fx["tembs"]) < 1e-3
    assert out.hidden_states_combineds is None and out.images == []


def test_tiny_injected_ratios_vs_golden(golden):
    pipe, inp, model = _tiny()
    fx = golden("tiny_traj")
    cu = {k: v.cuda() for k, v in inp.items()}
    out = model(**cu, max_inference_steps=8, predict=False, ratios=fx["sample.ratios"])
    assert float((out.sigmas.cpu() - fx["sample.sigmas"]).abs().max()) < 1e-5       # sigma_next = sigma * injected ratio
    assert float((out.logprobs.cpu() - fx["sample.logprobs"]).abs().max()) < 2e-2
    assert rel(out.latents, fx["sample.final_latents"]) < LATENT_TOL
    # replay (only_predict_logprobs) reproduces the rollout log-probs from the recorded TPM inputs
    assert out.hidden_states_combineds.shape == (2, 8, 768, 16, 16)
    lp = model.only_predict_logprobs(out.sigmas, out.hidden_states_combineds, out.tembs)["logprobs"]
    assert float((lp - out.logprobs).abs().max()) < 2e-3
    with pytest.raises(ValueError):
        model.only_predict_logprobs(None, None, None)


@pytest.mark.parametrize("predict", [True, False])
def test_graph_replayed_steps_equal_plain_steps(predict):
    """Engine.sample replays every step index from a CUDA graph (tpdm_sample_step_graph).  Capture (first trajectory), replay (second
    trajectory, other latents and guidance -> graphs dropped and re-captured; third: pure replay) and the plain launch path must give
    bit-identical trajectories; injected ratios go through the graphs too, device-side draws (seed argument) take the plain path."""
    pipe, inp, model = _tiny()
    eng = model.get_engine()
    g = torch.Generator().manual_seed(5)
    cu = {k: v.cuda() for k, v in inp.items()}
    args = (cu["prompt_embeds"], cu["negative_prompt_embeds"], cu["pooled_prompt_embeds"], cu["negative_pooled_prompt_embeds"])
    ratios = None if predict else (0.55 + 0.4 * torch.rand(2, 8, generator=g)).cuda()
    keys = ("sigmas", "alphas", "betas", "logprobs_raw", "history_latents", "tembs")
    for trial, (gs, lat) in enumerate(((7.0, cu["latents"]), (3.5, cu["latents"] * 0.5 + 0.1), (3.5, cu["latents"].flip(0)))):
        runs = [eng.sample(lat, *args, 8, gs, predict, ratios=ratios, record_velocity=True, use_graph=ug) for ug in (True, False, True)]
        for k in keys + ("velocities",):
            assert torch.equal(runs[0][k], runs[1][k]) and torch.equal(runs[2][k], runs[1][k]), (trial, k)
        assert runs[0]["steps"] == runs[1]["steps"]
    # device-side Beta draws: same seed -> same trajectory with and without use_graph (both run the plain step)
    a = eng.sample(cu["latents"], *args, 6, 7.0, False, seed=11, use_graph=True)
    b = eng.sample(cu["latents"], *args, 6, 7.0, False, seed=11, use_graph=False)
    assert torch.equal(a["sigmas"], b["sigmas"]) and torch.equal(a["history_latents"], b["history_latents"])


def test_tiny_early_termination_and_device_sampler():
    """min_sigma high enough that the batch finishes before max steps: loop must stop exactly like the reference
    (one masked step after sigma < min_sigma) and device-side Beta draws must be valid and seed-reproducible."""
    pipe, inp, model = _tiny()
    model.min_sigma = 0.2
    pipe.min_sigma = 0.2
    cu = {k: v.cuda() for k, v in inp.items()}
    ref = pipe(**inp, max_inference_steps=28, predict=True)
    out = model(**cu, max_inference_steps=28, predict=True)
    assert out.sigmas.shape == ref["sigmas"].shape
    assert float((out.sigmas.cpu() - ref["sigmas"]).abs().max()) < SIGMA_TOL
    assert torch.equal(out.prob_masks.cpu(), ref["prob_masks"])
    assert rel(out.latents, ref["final_latents"]) < LATENT_TOL
    g = torch.Generator().manual_seed(3)
    a = model(**cu, max_inference_steps=6, predict=False, generator=g)
    b = model(**cu, max_inference_steps=6, predict=False, generator=torch.Generator().manual_seed(3))
    assert torch.equal(a.sigmas, b.sigmas)
    r = a.sigmas[:, 0]
    assert bool(((r > 0) & (r < 1)).all()) and float(a.sigmas.std()) > 0


# ---------------------------------------------------------------------------------------------------------------
# SD3-medium shapes (BASELINE.json configs[1]): one MMDiT forward vs the fp32 oracle on the GPU (TF32 off)
# ---------------------------------------------------------------------------------------------------------------
def test_mmdit_forward_sd3_medium_1024_vs_oracle():
    from oracle import sd3_oracle as O
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = O.sd3_medium_config()
    torch.manual_seed(1234)
    with torch.device("cuda"):
        ora = O.OracleSD3Transformer(cfg).requires_grad_(False).eval()
    ora = ora.to("cuda")    # the sincos buffer is built with numpy on the host
    model =CustomSD3Transformer2DModel(sample_size=128, num_layers=24, attention_head_dim=64, num_attention_heads=24,
                                        caption_projection_dim=1536, pos_embed_max_size=192, device="cuda", dtype=torch.bfloat16)
    model.load_state_dict(ora.state_dict())
    ora.load_state_dict(model.state_dict())     # both sides see the same bf16-representable weights
    g = torch.Generator(device="cuda").manual_seed(0)
    lat = torch.randn(1, 16, 128, 128, device="cuda", generator=g).repeat(2, 1, 1, 1)
    enc = torch.randn(2, 333, 4096, device="cuda", generator=g)
    pooled = torch.randn(2, 2048, device="cuda", generator=g)
    ts = torch.tensor([700.0, 700.0], device="cuda")
    with torch.no_grad():
        rv, rt, rh1, rh2 = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat.float(), enc, pooled, ts, return_dict=False)
    assert rel(temb, rt) < 2e-3
    assert rel(h1, rh1) < 1e-3
    assert rel(h2, rh2) < VEL_TOL
    assert rel(v, rv) < VEL_TOL


# ---------------------------------------------------------------------------------------------------------------
# other BASELINE.json configs as parity cases (reduced depth keeps the fp32 oracle cheap; widths / sequence lengths are
# the real ones) and size-independent properties at full size
# ---------------------------------------------------------------------------------------------------------------
def _sd3m_pair(num_layers, sample_size, qk_norm=None):
    from oracle import sd3_oracle as O
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = O.sd3_medium_config(sample_size=sample_size, qk_norm=qk_norm)
    cfg.num_layers = num_layers
    torch.manual_seed(4321)
    ora = O.OracleSD3Transformer(cfg).requires_grad_(False).eval().to("cuda")
    model = CustomSD3Transformer2DModel(sample_size=sample_size, num_layers=num_layers, attention_head_dim=64, num_attention_heads=24,
                                        caption_projection_dim=1536, pos_embed_max_size=192, qk_norm=qk_norm, device="cuda",
                                        dtype=torch.bfloat16)
    model.load_state_dict(ora.state_dict())
    ora.load_state_dict(model.state_dict())
    return ora, model


def test_mmdit_2048_long_sequence_vs_oracle():
    """BASELINE config 5: 16 384 image tokens + 333 text tokens (S = 16 717), batch 1 with CFG (Bt = 2)."""
    ora, model = _sd3m_pair(num_layers=2, sample_size=256)
    g = torch.Generator(device="cuda").manual_seed(2)
    lat = torch.randn(1, 16, 256, 256, device="cuda", generator=g).repeat(2, 1, 1, 1)
    enc = torch.randn(2, 333, 4096, device="cuda", generator=g)
    pooled = torch.randn(2, 2048, device="cuda", generator=g)
    ts = torch.tensor([400.0, 400.0], device="cuda")
    with torch.no_grad():
        rv, rt, rh1, rh2 = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat, enc, pooled, ts, return_dict=False)
    assert v.shape == (2, 16, 256, 256)
    assert rel(h2, rh2) < VEL_TOL and rel(v, rv) < VEL_TOL


def test_mmdit_512_batch32_qknorm_vs_oracle():
    """BASELINE config 4 shape: 512^2, 16 rollouts with CFG -> transformer batch 32; QK-RMSNorm on."""
    ora, model = _sd3m_pair(num_layers=2, sample_size=64, qk_norm="rms_norm")
    g = torch.Generator(device="cuda").manual_seed(3)
    lat = torch.randn(32, 16, 64, 64, device="cuda", generator=g)
    enc = torch.randn(32, 333, 4096, device="cuda", generator=g)
    pooled = torch.randn(32, 2048, device="cuda", generator=g)
    ts = torch.rand(32, device="cuda", generator=g) * 1000
    with torch.no_grad():
        rv, rt, rh1, rh2 = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat, enc, pooled, ts, return_dict=False)
    assert rel(temb, rt) < 2e-3 and rel(h2, rh2) < VEL_TOL and rel(v, rv) < VEL_TOL


def test_attention_full_size_properties(L):
    """S = 4429, H = 24 (SD3-medium 1024^2): rows of softmax sum to one (V = 1 -> O = 1) and the result does not depend
    on the order of the keys."""
    torch.manual_seed(6)
    lib = L.load()
    Bt, S, H, d = 1, 4429, 24, 64
    qkv = torch.randn(Bt, S, 3, H, d, device="cuda").bfloat16()
    ones = qkv.clone()
    ones[:, :, 2] = 1.0
    out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
    L.check(lib.tpdm_joint_attention(L.ptr(ones), L.ptr(out), Bt, S, H, 64, d, 0, None))
    torch.cuda.synchronize()
    assert float((out.float() - 1.0).abs().max()) < 1e-2
    base = torch.zeros_like(out)
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(base), Bt, S, H, 64, d, 0, None))
    perm = torch.randperm(S, device="cuda")
    shuffled = qkv.clone()
    shuffled[:, :, 1:] = qkv[:, perm, 1:]          # permute keys and values together, queries stay
    out2 = torch.zeros_like(out)
    L.check(lib.tpdm_joint_attention(L.ptr(shuffled.contiguous()), L.ptr(out2), Bt, S, H, 64, d, 0, None))
    torch.cuda.synchronize()
    assert rel(out2, base) < 6e-3


def test_gemm_linearity_full_size(L):
    """QKV shape of SD3-medium 1024^2: A (W1 + W2)^T == A W1^T + A W2^T within bf16 rounding of the weights."""
    torch.manual_seed(7)
    lib = L.load()
    A = (torch.randn(2, 4096, 1536, device="cuda") * 0.5).bfloat16()
    W1 = (torch.randn(4608, 1536, device="cuda") * 0.03).bfloat16()
    W2 = (torch.randn(4608, 1536, device="cuda") * 0.03).bfloat16()
    Ws = (W1.float() + W2.float()).bfloat16()
    outs = []
    for W in (W1, W2, Ws):
        o = torch.zeros(2, 4096, 4608, device="cuda")
        L.check(lib.tpdm_gemm_bf16(L.ptr(A), L.ptr(W), None, None, L.ptr(o), 2, 4096, 4608, 1536, 1, None))
        outs.append(o)
    torch.cuda.synchronize()
    assert rel(outs[0] + outs[1], outs[2]) < 4e-3


def test_sd3_medium_trajectory_is_deterministic_and_terminates():
    """BASELINE config 1 at full size: the loop stops by itself (sigma_next < min_sigma), one masked step after sigma falls
    below min_sigma exactly as the reference does, and two runs are bit-identical."""
    from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel

    torch.manual_seed(11)
    model = SD3PredictNextTimeStepModel(transformer_config=SD3_MEDIUM_TRANSFORMER_CONFIG, torch_dtype=torch.bfloat16, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    kw = dict(prompt_embeds=torch.randn(1, 333, 4096, device="cuda", generator=g),
              negative_prompt_embeds=torch.randn(1, 333, 4096, device="cuda", generator=g),
              pooled_prompt_embeds=torch.randn(1, 2048, device="cuda", generator=g),
              negative_pooled_prompt_embeds=torch.randn(1, 2048, device="cuda", generator=g),
              latents=torch.randn(1, 16, 128, 128, device="cuda", generator=g))
    a = model(**kw, max_inference_steps=28, predict=True)
    b = model(**kw, max_inference_steps=28, predict=True)
    T = a.sigmas.shape[1]
    assert 10 < T < 28
    assert torch.equal(a.sigmas, b.sigmas) and torch.equal(a.latents, b.latents)
    sig = a.sigmas[0].cpu()
    assert bool((sig[:-1] > sig[1:]).all()) and float(sig[-1]) < model.min_sigma
    assert torch.isfinite(a.latents).all() and torch.isfinite(a.logprobs).all()
    alpha, beta = a.alphas[0, 0].item(), a.betas[0, 0].item()
    assert abs(float(sig[0]) - (alpha - 1) / (alpha + beta - 2)) < 1e-5     # first step: sigma_1 = 1 * Beta mode


@pytest.mark.parametrize("qk_norm,dual", [("rms_norm", (0, 1, 2)), (None, (1,))])
def test_mmdit_sd35_dual_attention_blocks_vs_oracle(qk_norm, dual):
    """SURVEY 8(f) rank 4 -- SD3.5 blocks (transformer_sd3.py:104-106,138): 9-chunk norm1, attn2 = image-token self-attention
    added after the joint attention, optionally QK-RMSNorm; SD3-medium width, 512^2, mixed dual / plain layers incl. the
    context_pre_only last block."""
    from oracle import sd3_oracle as O
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = O.sd3_medium_config(sample_size=64, qk_norm=qk_norm)
    cfg.num_layers = 3
    cfg.dual_attention_layers = dual
    torch.manual_seed(99)
    ora = O.OracleSD3Transformer(cfg).requires_grad_(False).eval().to("cuda")
    model = CustomSD3Transformer2DModel(sample_size=64, num_layers=3, attention_head_dim=64, num_attention_heads=24, caption_projection_dim=1536,
                                        pos_embed_max_size=192, qk_norm=qk_norm, dual_attention_layers=dual, device="cuda", dtype=torch.bfloat16)
    model.load_state_dict(ora.state_dict())
    ora.load_state_dict(model.state_dict())
    g = torch.Generator(device="cuda").manual_seed(5)
    lat = torch.randn(2, 16, 64, 64, device="cuda", generator=g)
    enc = torch.randn(2, 333, 4096, device="cuda", generator=g)
    pooled = torch.randn(2, 2048, device="cuda", generator=g)
    ts = torch.tensor([250.0, 800.0], device="cuda")
    with torch.no_grad():
        rv, rt, rh1, rh2 = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat, enc, pooled, ts, return_dict=False)
    assert rel(temb, rt) < 2e-3 and rel(h2, rh2) < VEL_TOL and rel(v, rv) < VEL_TOL
    # the attn2 branch really contributes: the same weights with attn2 ignored give a different answer
    cfg0 = O.sd3_medium_config(sample_size=64, qk_norm=qk_norm)
    cfg0.num_layers = 3
    plain = O.OracleSD3Transformer(cfg0).requires_grad_(False).eval().to("cuda")
    sd = {k: (t[: plain.state_dict()[k].shape[0]] if "norm1.linear" in k else t) for k, t in ora.state_dict().items() if k in plain.state_dict()}
    plain.load_state_dict(sd)
    with torch.no_grad():
        pv = plain(lat, enc, pooled, ts)[0]
    assert rel(pv, rv) > 5 * rel(v, rv)


def test_device_prompt_queue_matches_per_prompt_sampling():
    """BASELINE config 3 mechanism: 7 prompts with different trajectory lengths through 3 in-flight slots refilled on the
    device == each prompt sampled alone (batch 1, predict=True): same step counts, same sigma sequences, same final latents.
    Two 'GPUs' sharing one ticket counter split the list without overlap."""
    from oracle import sd3_oracle as O
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    tiny = dict(sample_size=32, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=96, num_attention_heads=4,
                joint_attention_dim=4096, caption_projection_dim=384, pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=96)
    torch.manual_seed(21)
    model = SD3PredictNextTimeStepModel(transformer_config=tiny, torch_dtype=torch.float32, device="cuda", min_sigma=0.05)
    with torch.no_grad():      # make the TimePredictor depend on its input so that trajectory lengths differ between prompts
        tp = model.time_predictor
        tp.fc2.weight.mul_(40)
        tp.fc1.weight.mul_(8)
        tp.conv2.weight.mul_(6)
        tp.norm1.linear.weight.mul_(4)
    P, T = 7, 12
    g = torch.Generator().manual_seed(3)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    pe, ne, pp, npp, lat = mk(P, 333, 4096), mk(P, 333, 4096), mk(P, 2048), mk(P, 2048), mk(P, 16, 32, 32)
    lat = lat * torch.linspace(0.5, 2.0, P, device="cuda").view(P, 1, 1, 1)     # different inputs -> different alpha/beta
    ref_steps, ref_lat, ref_sig = [], [], []
    for i in range(P):
        o = model(prompt_embeds=pe[i:i + 1], negative_prompt_embeds=ne[i:i + 1], pooled_prompt_embeds=pp[i:i + 1],
                  negative_pooled_prompt_embeds=npp[i:i + 1], latents=lat[i:i + 1], max_inference_steps=T, predict=True)
        ref_steps.append(o.sigmas.shape[1])
        ref_lat.append(o.latents[0])
        ref_sig.append(o.sigmas[0])
    assert len(set(ref_steps)) > 1, ref_steps          # the stress is real: lengths differ
    q = model.sample_queue(pe, ne, pp, npp, latents=lat, slots=3, max_inference_steps=T)     # CUDA-graph replay of the step
    q_eager = model.sample_queue(pe, ne, pp, npp, latents=lat, slots=3, max_inference_steps=T, use_graph=False)
    assert q_eager.steps.tolist() == ref_steps and rel(q_eager.latents, q.latents) < 1e-6
    assert q.steps.tolist() == ref_steps
    for i in range(P):
        n = ref_steps[i]
        assert torch.allclose(q.sigmas[i, 1:n + 1], ref_sig[i], atol=1e-5)
        assert rel(q.latents[i], ref_lat[i]) < 1e-4
    # longest-expected-first scheduling (one probe step per prompt, tickets sorted by the expected length): same trajectories
    q_lpt = model.sample_queue(pe, ne, pp, npp, latents=lat, slots=3, max_inference_steps=T, schedule="lpt")
    assert q_lpt.steps.tolist() == ref_steps
    for i in range(P):
        n = ref_steps[i]
        assert torch.allclose(q_lpt.sigmas[i, 1:n + 1], ref_sig[i], atol=1e-5)
        assert rel(q_lpt.latents[i], ref_lat[i]) < 1e-4
    assert q_lpt.device_steps <= q.device_steps + 1
    # fewer device steps than running the prompts one after the other, and no more than slots allow
    assert q.device_steps < sum(ref_steps) and q.device_steps >= -(-sum(ref_steps) // 3)
    # two workers sharing one ticket counter: every prompt is processed exactly once
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    a = model.sample_queue(pe, ne, pp, npp, latents=lat, slots=2, max_inference_steps=T, ticket=ticket)
    assert int(ticket) >= P and a.steps.tolist() == ref_steps     # a single worker drains the shared counter completely
    ticket.zero_()
    ticket += 4                                                   # another worker already took prompts 0..3
    b = model.sample_queue(pe, ne, pp, npp, latents=lat, slots=2, max_inference_steps=T, ticket=ticket)
    assert b.steps.tolist() == [0, 0, 0, 0] + ref_steps[4:]
    with pytest.raises(ValueError):
        model.sample_queue(pe, ne, pp, npp, latents=lat, slots=P + 1, max_inference_steps=T)


def test_mmdit_sd35_large_width_vs_oracle():
    """SD3.5-large block shape (38 heads x 64 = 2432 wide, QK-RMSNorm): hidden sizes that are not multiples of the 256-wide
    GEMM tile (N tails in every projection) and take the generic LayerNorm path; 2 layers, 512^2."""
    from oracle import sd3_oracle as O
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = O.SD3Config(sample_size=64, num_layers=2, attention_head_dim=64, num_attention_heads=38, caption_projection_dim=2432,
                      pos_embed_max_size=192, qk_norm="rms_norm")
    torch.manual_seed(77)
    ora = O.OracleSD3Transformer(cfg).requires_grad_(False).eval().to("cuda")
    model = CustomSD3Transformer2DModel(sample_size=64, num_layers=2, attention_head_dim=64, num_attention_heads=38, caption_projection_dim=2432,
                                        pos_embed_max_size=192, qk_norm="rms_norm", device="cuda", dtype=torch.bfloat16)
    model.load_state_dict(ora.state_dict())
    ora.load_state_dict(model.state_dict())
    g = torch.Generator(device="cuda").manual_seed(8)
    lat = torch.randn(2, 16, 64, 64, device="cuda", generator=g)
    enc = torch.randn(2, 333, 4096, device="cuda", generator=g)
    pooled = torch.randn(2, 2048, device="cuda", generator=g)
    ts = torch.tensor([100.0, 900.0], device="cuda")
    with torch.no_grad():
        rv, rt, rh1, rh2 = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat, enc, pooled, ts, return_dict=False)
    assert rel(temb, rt) < 2e-3 and rel(h1, rh1) < 1e-3 and rel(h2, rh2) < VEL_TOL and rel(v, rv) < VEL_TOL


def test_ln_modulate_full_size_properties(L):
    """SD3-medium block shape (2 x 4096 rows of 1536): with zero shift / scale every output row is standardised; a constant
    shift moves the row mean, a constant scale the row spread; rows do not influence each other (permutation equivariance)."""
    torch.manual_seed(12)
    lib = L.load()
    B, rows, D = 2, 4096, 1536
    x = torch.randn(B, rows, D, device="cuda") * torch.rand(B, rows, 1, device="cuda").mul(5).add(0.1) + torch.randn(B, rows, 1, device="cuda") * 4
    out = torch.empty(B, rows, D, device="cuda", dtype=torch.bfloat16)

    def run(inp, mod):
        L.check(lib.tpdm_ln_modulate(L.ptr(inp), mod.data_ptr(), mod.data_ptr() + 4 * D, 2 * D, L.ptr(out), B, rows, D, None))
        torch.cuda.synchronize()
        return out.float().clone()

    zero = torch.zeros(B, 2 * D, device="cuda")
    y = run(x, zero)
    assert float(y.mean(-1).abs().max()) < 2e-2 and float((y.var(-1, unbiased=False) - 1).abs().max()) < 2e-2
    mod = zero.clone()
    mod[:, :D] = 0.75       # shift
    mod[:, D:] = 1.0        # scale -> factor 2
    y2 = run(x, mod)
    assert float((y2.mean(-1) - 0.75).abs().max()) < 3e-2 and float((y2.var(-1, unbiased=False) - 4).abs().max()) < 8e-2
    perm = torch.randperm(rows, device="cuda")
    yp = run(x[:, perm].contiguous(), zero)
    assert torch.equal(yp, y[:, perm])


def test_euler_step_round_trip_full_size():
    """custom_step at the 1024^2 latent shape: stepping sigma -> sigma_next and back returns the sample (fp32 rounding only), and
    the step is linear in the model output."""
    from tpdm_b200.model_utilis import CustomFlowMatchEulerDiscreteScheduler

    sch = CustomFlowMatchEulerDiscreteScheduler()
    g = torch.Generator(device="cuda").manual_seed(13)
    x = torch.randn(2, 16, 128, 128, device="cuda", generator=g)
    v = torch.randn(2, 16, 128, 128, device="cuda", generator=g)
    s0, s1 = torch.tensor([1.0, 0.62], device="cuda"), torch.tensor([0.71, 0.40], device="cuda")
    fwd = sch.custom_step(v, s1, s0, x, return_dict=False)[0]
    back = sch.custom_step(v, s0, s1, fwd, return_dict=False)[0]
    assert float((back - x).abs().max()) < 1e-5
    assert torch.allclose(fwd, x + (s1 - s0).view(-1, 1, 1, 1) * v, atol=1e-6)
    twice = sch.custom_step(2 * v, s1, s0, x, return_dict=False)[0]
    assert torch.allclose(twice - x, 2 * (fwd - x), atol=1e-5)
