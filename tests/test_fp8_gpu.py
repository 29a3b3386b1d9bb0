"""The opt-in FP8 (E4M3) mode of the MMDiT's QKV and FF1 projections (run with -m gpu on a B200): the row quantizer, the FP8
LN-modulate and the FP8 CTA-pair GEMM through their C-ABI entries, then the MMDiT forward and a closed-loop trajectory
against the oracle with the same fake quantization (tests/fp8_fake_quant.py), and the sampler surfaces in FP8
mode.  Velocity bar against the fake-quant oracle: 2e-2 rel-L2, the bar the bf16 path meets against the fp32 oracle; against
the plain fp32 oracle the error is printed and held to 4e-2."""
import pytest
import torch

from kernel_check import assert_launch, gemm_magnitude, guarded

pytestmark = pytest.mark.gpu

VEL_TOL, PLAIN_VEL_TOL, SIGMA_TOL, LATENT_TOL = 2e-2, 4e-2, 1e-3, 3e-2
TINY = dict(sample_size=32, num_layers=2, attention_head_dim=96, num_attention_heads=4, caption_projection_dim=384, pos_embed_max_size=96)


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")


@pytest.fixture(scope="module")
def L():
    from tpdm_b200 import _lib

    _lib.load()
    return _lib


def _quantize(L, x):
    lib = L.load()
    x = x.float().contiguous()
    codes = torch.empty(x.shape, dtype=torch.uint8, device="cuda")
    scales = torch.empty(x.shape[:-1], dtype=torch.float32, device="cuda")
    L.check(lib.tpdm_quantize_fp8_rows(L.ptr(x), x.numel() // x.shape[-1], x.shape[-1], L.ptr(codes), L.ptr(scales), None))
    torch.cuda.synchronize()
    return codes, scales


# ---------------------------------------------------------------------------------------------------------------
# unit kernels
# ---------------------------------------------------------------------------------------------------------------
def test_quantize_rows_matches_torch_bit_for_bit(L):
    from fp8_fake_quant import quantize_e4m3_rows

    g = torch.Generator().manual_seed(0)
    K = 1536
    rows = [torch.randn(64, K, generator=g) * 0.05,                               # ordinary weight rows
            torch.randn(16, K, generator=g) * 0.01,                               # one large outlier per row: the rest lands on
            torch.randn(16, K, generator=g) * 1e-20,                              # E4M3 subnormals; tiny (normal fp32) rows
            torch.zeros(4, K)]                                                    # zero rows: scale 1, zero codes
    rows[1][torch.arange(16), torch.randint(0, K, (16,), generator=g)] = 30.0
    x = torch.cat(rows)
    codes, scales = _quantize(L, x.cuda())
    ref_codes, ref_scales = quantize_e4m3_rows(x)
    assert torch.equal(codes.cpu(), ref_codes.view(torch.uint8))
    assert torch.equal(scales.cpu(), ref_scales)
    sub = ref_codes[64:80].float().abs()
    assert bool(((sub > 0) & (sub < 2 ** -6)).any())                               # the outlier rows do exercise subnormal codes
    assert bool((scales[-4:] == 1).all()) and int(codes[-4:].sum()) == 0


@pytest.mark.parametrize("D", [1536, 384, 512])
def test_ln_modulate_fp8_matches_torch(L, D):
    from fp8_fake_quant import quantize_e4m3_rows

    lib = L.load()
    torch.manual_seed(1)
    B, rows, R = 2, 333, 3 * D
    x = torch.randn(B, rows, D, device="cuda") * 3 + 0.5
    mod = torch.randn(B, R, device="cuda") * 0.5
    shift, scale = mod[:, :D], mod[:, D: 2 * D]
    codes = torch.empty(B, rows, D, dtype=torch.uint8, device="cuda")
    sc = torch.empty(B, rows, device="cuda")
    L.check(lib.tpdm_ln_modulate_fp8(L.ptr(x), L.ptr(mod), mod.data_ptr() + 4 * D, R, L.ptr(codes), L.ptr(sc), B, rows, D, None))
    torch.cuda.synchronize()
    y = torch.nn.functional.layer_norm(x, (D,), eps=1e-6) * (1 + scale[:, None]) + shift[:, None]
    rc, rs = quantize_e4m3_rows(y.cpu())
    rc = rc.view(torch.uint8)
    c = codes.cpu()
    same = (c == rc).float().mean().item()
    mag = lambda t: (t & 0x7F).int()
    apart = ((mag(c) - mag(rc)).abs() <= 1) & ((c & 0x80) == (rc & 0x80)) | ((mag(c) <= 1) & (mag(rc) <= 1))
    print(f"[ln_modulate fp8 D={D}] identical codes {same:.5f}")
    assert same >= 0.999 and bool(apart.all())
    assert float(((sc.cpu() - rs).abs() / rs).max()) <= 1e-6


GEMM_SHAPES = [   # (batch, rows, N, K, epi): SD3-M QKV image rows and text tail, FF1 + GELU, tiny config, K = 2432 (19 k-blocks)
    (2, 4096, 4608, 1536, 0), (2, 333, 4608, 1536, 0), (2, 4096, 6144, 1536, 2), (2, 333, 1152, 384, 0), (2, 512, 7296, 2432, 0),
    (32, 333, 4608, 1536, 0), (32, 256, 6144, 1536, 2), (2, 4096, 4608, 1536, 1), (2, 333, 6144, 1536, 1), (32, 333, 1152, 384, 1),
    (2, 512, 7296, 2432, 1)]


@pytest.mark.parametrize("batch,rows,N,K,epi", GEMM_SHAPES)
def test_gemm_fp8_vs_dequantized_fp32(L, batch, rows, N, K, epi):
    """every element against the float64 product of the dequantized operands (tests/kernel_check.py); nothing written outside
    [batch][rows][N]"""
    lib = L.load()
    torch.manual_seed(2)
    A = torch.randn(batch, rows, K, device="cuda")
    W = torch.randn(N, K, device="cuda") * 0.03
    bias = torch.randn(N, device="cuda") * 0.1
    a8, a_s = _quantize(L, A)
    w8, w_s = _quantize(L, W)
    deq = lambda c, s: c.view(torch.float8_e4m3fn).double() * s.double().unsqueeze(-1)
    a64, w64 = deq(a8, a_s), deq(w8, w_s)
    pre = a64 @ w64.t() + bias.double()
    mag = gemm_magnitude(a64, w64, bias)
    buf, out = guarded((batch, rows, N), torch.float32 if epi == 1 else torch.bfloat16)
    ref = torch.nn.functional.gelu(pre, approximate="tanh") if epi == 2 else pre
    before = buf.clone()
    L.check(lib.tpdm_gemm_fp8(L.ptr(a8), L.ptr(a_s), L.ptr(w8), L.ptr(w_s), L.ptr(bias), L.ptr(out), batch, rows, N, K, epi, None))
    torch.cuda.synchronize()
    assert_launch(buf, before, [(out, ref, mag, pre if epi == 2 else None)], what=f"gemm fp8 {batch}x{rows}x{N}x{K} epi {epi}")


def test_gemm_fp8_rejects_bad_arguments(L):
    lib = L.load()
    a8 = torch.zeros(1, 8, 64, dtype=torch.uint8, device="cuda")
    w8 = torch.zeros(128, 64, dtype=torch.uint8, device="cuda")
    s = torch.ones(128, device="cuda")
    out = torch.zeros(1, 8, 128, device="cuda")
    with pytest.raises(ValueError):          # N = 128 has no CTA-pair tile
        L.check(lib.tpdm_gemm_fp8(L.ptr(a8), L.ptr(s), L.ptr(w8), L.ptr(s), None, L.ptr(out), 1, 8, 128, 64, 1, None))
    with pytest.raises(ValueError):          # the gate epilogue has no FP8 form
        L.check(lib.tpdm_gemm_fp8(L.ptr(a8), L.ptr(s), L.ptr(w8), L.ptr(s), None, L.ptr(out), 1, 8, 256, 64, 3, None))


# ---------------------------------------------------------------------------------------------------------------
# MMDiT forward against the fake-quant oracle
# ---------------------------------------------------------------------------------------------------------------
def _forward_pair(cfg, model_kw, seed, sample, batch=2, t=400.0):
    from fp8_fake_quant import set_fp8_fake_quant
    from oracle import sd3_oracle as O
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    _no_tf32()
    torch.manual_seed(seed)
    ora = O.OracleSD3Transformer(cfg).requires_grad_(False).eval().to("cuda")
    model = CustomSD3Transformer2DModel(**model_kw, device="cuda", dtype=torch.bfloat16, mmdit_precision="fp8")
    model.load_state_dict(ora.state_dict())
    ora.load_state_dict(model.state_dict())
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    lat = torch.randn(batch, 16, sample, sample, device="cuda", generator=g)
    enc = torch.randn(batch, 333, cfg.joint_attention_dim, device="cuda", generator=g)
    pooled = torch.randn(batch, cfg.pooled_projection_dim, device="cuda", generator=g)
    ts = torch.full((batch,), t, device="cuda")
    with torch.no_grad():
        plain = ora(lat, enc, pooled, ts)
        set_fp8_fake_quant(ora)
        fq = ora(lat, enc, pooled, ts)
    v, temb, h1, h2 = model(lat, enc, pooled, ts, return_dict=False)
    return (v, h2), (fq[0], fq[3]), (plain[0], plain[3])


@pytest.mark.parametrize("case", ["sd3m_1024", "tiny", "tiny_qknorm", "tiny_dual"])
def test_mmdit_forward_fp8_vs_fake_quant_oracle(case):
    from oracle import sd3_oracle as O

    if case == "sd3m_1024":
        cfg = O.sd3_medium_config(sample_size=128)
        kw = dict(sample_size=128, num_layers=24, attention_head_dim=64, num_attention_heads=24, caption_projection_dim=1536,
                  pos_embed_max_size=192)
        sample = 128
    else:
        cfg = O.tiny_config(qk_norm="rms_norm" if case == "tiny_qknorm" else None)
        kw = dict(TINY, qk_norm=cfg.qk_norm)
        if case == "tiny_dual":
            cfg.dual_attention_layers = (0,)
            kw["dual_attention_layers"] = (0,)
        sample = 32
    (v, h2), (fv, fh2), (pv, ph2) = _forward_pair(cfg, kw, 4321, sample)
    ev, eh, pv_e = rel(v, fv), rel(h2, fh2), rel(v, pv)
    print(f"[fp8 forward {case}] velocity rel-L2 vs fake-quant oracle {ev:.2e} (h2 {eh:.2e}); vs plain fp32 oracle {pv_e:.2e} "
          f"(h2 {rel(h2, ph2):.2e}); fake-quant vs plain oracle {rel(fv, pv):.2e}")
    assert ev <= VEL_TOL and eh <= VEL_TOL
    assert pv_e <= PLAIN_VEL_TOL


def test_closed_loop_1024_reference_init_vs_fake_quant_oracle():
    from fp8_fake_quant import set_fp8_fake_quant
    from oracle import sd3_oracle as O
    from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel

    _no_tf32()
    cfg = O.sd3_medium_config(sample_size=128)
    torch.manual_seed(1234)
    pipe = O.OraclePipeline(cfg).to("cuda")
    model = SD3PredictNextTimeStepModel(transformer_config=dict(SD3_MEDIUM_TRANSFORMER_CONFIG), torch_dtype=torch.bfloat16, device="cuda",
                                        mmdit_precision="fp8")
    model.transformer.load_state_dict(pipe.transformer.state_dict())
    model.time_predictor.load_state_dict(pipe.time_predictor.state_dict())
    pipe.transformer.load_state_dict(model.transformer.state_dict())
    pipe.time_predictor.load_state_dict(model.time_predictor.state_dict())
    set_fp8_fake_quant(pipe.transformer)
    g = torch.Generator(device="cuda").manual_seed(3)
    mk = lambda *s: torch.randn(*s, device="cuda", generator=g)
    kw = dict(prompt_embeds=mk(1, 333, 4096), negative_prompt_embeds=mk(1, 333, 4096), pooled_prompt_embeds=mk(1, 2048),
              negative_pooled_prompt_embeds=mk(1, 2048), latents=mk(1, 16, 128, 128))
    ref = pipe(**kw, max_inference_steps=28, predict=True, record_velocity=True)
    out = model(**kw, max_inference_steps=28, predict=True, return_velocities=True)
    T, T_ref = out.sigmas.shape[1], ref["sigmas"].shape[1]
    n = min(T, T_ref)
    dsig = float((out.sigmas[:, :n].float().cpu() - ref["sigmas"][:, :n].float().cpu()).abs().max())
    vel = [rel(out["velocities"][:, t], ref["velocities"][:, t]) for t in range(n)]
    dl = rel(out.latents, ref["final_latents"])
    print(f"[fp8 closed loop 1024] steps {T} / {T_ref}  max|dsigma| {dsig:.2e}  max velocity rel-L2 {max(vel):.2e}  final latent {dl:.2e}")
    assert T == T_ref and torch.equal(out.prob_masks.cpu(), ref["prob_masks"].cpu())
    assert dsig <= SIGMA_TOL and max(vel) <= VEL_TOL and dl <= LATENT_TOL


# ---------------------------------------------------------------------------------------------------------------
# sampler surfaces in FP8 mode (tiny config)
# ---------------------------------------------------------------------------------------------------------------
def _tiny_model(precision, seed=21, min_sigma=0.05):
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    torch.manual_seed(seed)
    model = SD3PredictNextTimeStepModel(transformer_config=TINY, torch_dtype=torch.float32, device="cuda", min_sigma=min_sigma,
                                        mmdit_precision=precision)
    with torch.no_grad():      # an input-sensitive TimePredictor: trajectory lengths differ between prompts
        tp = model.time_predictor
        tp.fc2.weight.mul_(40)
        tp.fc1.weight.mul_(8)
        tp.conv2.weight.mul_(6)
        tp.norm1.linear.weight.mul_(4)
    return model


def _embeds(P, seed=3):
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    return dict(prompt_embeds=mk(P, 333, 4096), negative_prompt_embeds=mk(P, 333, 4096), pooled_prompt_embeds=mk(P, 2048),
                negative_pooled_prompt_embeds=mk(P, 2048), latents=mk(P, 16, 32, 32))


def _engine_sample(model, kw, use_graph, T=12, predict=True):
    eng = model.get_engine()
    return eng.sample(kw["latents"], kw["prompt_embeds"], kw["negative_prompt_embeds"], kw["pooled_prompt_embeds"],
                      kw["negative_pooled_prompt_embeds"], T, 7.0, predict, use_graph=use_graph)


def test_fp8_graph_replay_and_repeat_runs_are_bit_identical():
    model = _tiny_model("fp8")
    kw = _embeds(2)
    a = _engine_sample(model, kw, use_graph=False)
    b = _engine_sample(model, kw, use_graph=True)
    c = _engine_sample(model, kw, use_graph=True)
    for k in ("sigmas", "alphas", "betas", "history_latents", "tembs"):
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(b[k], c[k]), k
    assert a["steps"] == b["steps"] == c["steps"]


def test_fp8_sample_queue_gives_every_prompt_its_batch1_trajectory():
    model = _tiny_model("fp8")
    P = 5
    kw = _embeds(P, seed=4)
    q = model.sample_queue(kw["prompt_embeds"], kw["negative_prompt_embeds"], kw["pooled_prompt_embeds"], kw["negative_pooled_prompt_embeds"],
                           kw["latents"], slots=2, max_inference_steps=12)
    steps = []
    for p in range(P):
        one = {k: v[p: p + 1] for k, v in kw.items()}
        out = model(**one, max_inference_steps=12, predict=True)
        steps.append(int((~out.prob_masks).sum()))
        assert int(q.steps[p]) == steps[-1], p
        assert torch.allclose(q.sigmas[p, 1: steps[-1] + 1], out.sigmas[0, : steps[-1]], atol=1e-5), p
        assert rel(q.latents[p: p + 1], out.latents) < 1e-4, p
    assert len(set(steps)) > 1          # trajectories of different lengths: slots were refilled and emptied (batch mask)


def test_fp8_rloo_update_through_the_queue():
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModelRLOOWrapper
    from tpdm_b200.rloo import rloo_update
    from tpdm_b200.tpm_training import TimePredictorTrainer

    torch.manual_seed(3)
    w = SD3PredictNextTimeStepModelRLOOWrapper(transformer_config=TINY, torch_dtype=torch.float32, device="cuda", min_sigma=0.01,
                                               max_inference_steps=6, mmdit_precision="fp8")
    kw = _embeds(2, seed=0)
    data = dict(prompt=["a", "b"], **{k: v for k, v in kw.items() if k != "latents"})
    trainer = TimePredictorTrainer(w.agent_model.time_predictor, grid=16, max_samples=4 * 6, lr=1e-3)
    res = rloo_update(w, trainer, data, reward_fn=lambda lat, out: -(lat.float() ** 2).mean(dim=(1, 2, 3)), rloo_k=2, num_ppo_epochs=2,
                      micro_batch_size=2, slots=3)
    assert w.agent_model.get_engine().mmdit_precision == "fp8"
    assert len(res["logs"]) == 4 and all(torch.isfinite(torch.tensor(list(l.values()))).all() for l in res["logs"])
    assert bool(torch.isfinite(res["scores"]).all()) and bool(torch.isfinite(res["advantages"]).all())


def test_bf16_unchanged_by_fp8_engines_and_switching_back():
    kw = _embeds(2, seed=5)
    model = _tiny_model("bf16")
    before = model(**kw, max_inference_steps=8, predict=True)
    fp8 = _tiny_model("fp8")
    f = fp8(**kw, max_inference_steps=8, predict=True)
    after = model(**kw, max_inference_steps=8, predict=True)
    assert torch.equal(before.latents, after.latents) and torch.equal(before.sigmas, after.sigmas)
    assert not torch.equal(f.latents, before.latents)                 # the FP8 engine really ran another path
    fp8.mmdit_precision = "bf16"                                      # the same model switched back: a fresh bf16 engine
    back = fp8(**kw, max_inference_steps=8, predict=True)
    assert fp8.get_engine().mmdit_precision == "bf16"
    assert torch.equal(back.latents, before.latents) and torch.equal(back.sigmas, before.sigmas)


def test_set_fp8_weights_after_a_plan_is_a_state_error(L):
    import ctypes as C

    from tpdm_b200.engine import pack_fp8_blocks

    lib = L.load()
    model = _tiny_model("bf16")
    kw = _embeds(1, seed=6)
    model(**kw, max_inference_steps=2, predict=True)                  # builds the engine and a plan
    eng = model.get_engine()
    pack_fp8_blocks(eng.weights, model.transformer.state_dict(), model.transformer.config, eng.device)
    with pytest.raises(RuntimeError, match="plan"):
        L.check(lib.tpdm_set_fp8_weights(eng.ctx, eng.weights.fp8_blocks))
    st = lib.tpdm_set_fp8_weights(eng.ctx, eng.weights.fp8_blocks)
    assert st == L.TPDM_ERR_STATE
    again = model(**kw, max_inference_steps=2, predict=True)          # the ctx is unchanged and keeps running bf16
    assert again.sigmas.shape[1] >= 1
