"""Sampled RLOO rollouts through the device-side prompt queue (``sample_rollouts``, C ABI ``tpdm_queue_set_rollout``) against the
lockstep batch ``forward(predict=False)`` of all prompts: same step counts, Beta draws, per-step records and output container."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TINY = dict(sample_size=32, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=96, num_attention_heads=4, joint_attention_dim=4096,
            caption_projection_dim=384, pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=96)
P, SLOTS, T_MAX, MIN_SIGMA = 7, 3, 12, 0.05


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _model(prediction_type="alpha_beta", relative=True, sensitive=True):
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    torch.manual_seed(21)
    model = SD3PredictNextTimeStepModel(transformer_config=TINY, torch_dtype=torch.float32, device="cuda", min_sigma=MIN_SIGMA,
                                        relative=relative, prediction_type=prediction_type)
    if sensitive:
        with torch.no_grad():      # make the TimePredictor depend on its input so that trajectory lengths differ between prompts
            tp = model.time_predictor
            tp.fc2.weight.mul_(40)
            tp.fc1.weight.mul_(8)
            tp.conv2.weight.mul_(6)
            tp.norm1.linear.weight.mul_(4)
    return model


def _embeds():
    g = torch.Generator().manual_seed(3)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    return mk(P, 333, 4096), mk(P, 333, 4096), mk(P, 2048), mk(P, 2048)


def _lockstep(model, emb, **kw):
    pe, ne, pp, npp = emb
    return model(prompt_embeds=pe, negative_prompt_embeds=ne, pooled_prompt_embeds=pp, negative_pooled_prompt_embeds=npp,
                 max_inference_steps=T_MAX, predict=False, **kw)


def _assert_same_rollouts(q, ref):
    """The queue's rollouts equal the lockstep batch's on every unmasked step."""
    assert set(q.keys()) - {"steps", "device_steps"} == set(ref.keys())
    assert q.sigmas.shape == ref.sigmas.shape and q.sigmas.dtype == ref.sigmas.dtype
    assert torch.equal(q.prob_masks, ref.prob_masks)
    valid = ~ref.prob_masks
    assert q.steps.tolist() == valid.sum(1).tolist()
    assert torch.allclose(q.sigmas[valid], ref.sigmas[valid], atol=1e-5)
    for k in ("alphas", "betas", "logprobs"):
        assert q[k].shape == ref[k].shape and q[k].dtype == ref[k].dtype
        assert rel(q[k][valid], ref[k][valid]) < 1e-4, k
    assert torch.equal(q.logprobs[~valid], ref.logprobs[~valid])                  # INVALID_LOGPROB = 1.0 at masked steps
    assert q.tembs.shape == ref.tembs.shape and rel(q.tembs[valid], ref.tembs[valid]) < 1e-4
    hq, hr = q.hidden_states_combineds, ref.hidden_states_combineds
    assert hq.shape == hr.shape and hq.dtype == hr.dtype == torch.bfloat16
    assert rel(hq[valid], hr[valid]) < 1e-4
    assert q.latents.shape == ref.latents.shape and rel(q.latents, ref.latents) < 1e-4
    assert [int(i) for i in q.last_valid_indices] == [int(i) for i in ref.last_valid_indices]
    assert q.images == ref.images == []


@pytest.fixture(scope="module")
def device_draws():
    """One model, its embeddings, and the lockstep rollout of all P prompts with device Beta draws."""
    model = _model()
    emb = _embeds()
    ref = _lockstep(model, emb, generator=torch.Generator().manual_seed(7))
    return model, emb, ref


def test_device_draws_match_the_lockstep_batch(device_draws):
    model, emb, ref = device_draws
    steps = (~ref.prob_masks).sum(1)
    assert len(set(steps.tolist())) > 1, steps                 # the stress is real: lengths differ
    q = model.sample_rollouts(*emb, slots=SLOTS, max_inference_steps=T_MAX, generator=torch.Generator().manual_seed(7))
    _assert_same_rollouts(q, ref)
    assert rel(q.init_noise_latents, ref.init_noise_latents) == 0.0           # the generator gave the same initial noise
    assert q.device_steps < P * ref.sigmas.shape[1]


@pytest.mark.parametrize("prediction_type,relative", [("alpha_beta", True), ("mode_concentration", False)])
def test_injected_ratios_match_the_lockstep_batch(prediction_type, relative):
    # injected ratios fix the lengths; the input-sensitive head would push the mode / concentration transform into NaN log-probs
    model = _model(prediction_type, relative, sensitive=prediction_type == "alpha_beta")
    emb = _embeds()
    g = torch.Generator().manual_seed(11)
    base = torch.linspace(0.5, 0.85, P) if relative else torch.linspace(0.06, 0.2, P)
    ratios = (base[:, None] * (0.9 + 0.2 * torch.rand(P, T_MAX, generator=g))).cuda()
    lat = torch.randn(P, 16, 32, 32, generator=g).cuda()
    ref = _lockstep(model, emb, latents=lat, ratios=ratios)
    assert len(set((~ref.prob_masks).sum(1).tolist())) > 1
    assert torch.isfinite(ref.logprobs).all()
    q = model.sample_rollouts(*emb, latents=lat, slots=SLOTS, max_inference_steps=T_MAX, ratios=ratios)
    _assert_same_rollouts(q, ref)


def test_graph_replay_equals_plain_launches(device_draws):
    model, emb, _ = device_draws
    a = model.sample_rollouts(*emb, slots=SLOTS, max_inference_steps=T_MAX, generator=torch.Generator().manual_seed(9))
    b = model.sample_rollouts(*emb, slots=SLOTS, max_inference_steps=T_MAX, generator=torch.Generator().manual_seed(9), use_graph=False)
    assert torch.equal(a.steps, b.steps) and torch.equal(a.prob_masks, b.prob_masks)
    for k in ("sigmas", "alphas", "betas", "logprobs", "tembs", "hidden_states_combineds", "latents"):
        assert rel(a[k], b[k]) < 1e-6, k


def test_records_past_the_end_are_zero_and_ppo_matches_lockstep(device_draws):
    from tpdm_b200.rloo import shape_rollout
    from tpdm_b200.tpm_training import TimePredictorTrainer

    model, emb, ref = device_draws
    q = model.sample_rollouts(*emb, slots=SLOTS, max_inference_steps=T_MAX, generator=torch.Generator().manual_seed(7))
    masked = q.prob_masks
    assert bool(masked.any())
    for k in ("alphas", "betas", "tembs", "hidden_states_combineds"):
        assert torch.isfinite(q[k].float()).all(), k
        assert bool((q[k][masked] == 0).all()), k
    assert bool((q.sigmas[masked] == 0).all())
    T = q.sigmas.shape[1]
    tr = TimePredictorTrainer(model.time_predictor, grid=16, max_samples=P * T)
    adv = torch.linspace(0.2, 1.0, P, device="cuda")            # one sign: the loss stays away from 0, a relative bound is meaningful
    stats, grads = [], []
    for out in (ref, q):
        x = out.hidden_states_combineds.permute(0, 1, 3, 4, 2)
        st = tr.ppo_update(out.sigmas, out.logprobs, x, out.tembs, adv, min_sigma=model.min_sigma, epsilon=model.epsilon,
                           relative=model.relative, prediction_type=model.prediction_type, optimizer_step=False)
        stats.append({k: v.clone() for k, v in st.items()})
        grads.append(tr.grads.clone())
    assert torch.isfinite(grads[1]).all() and float(grads[0].norm()) > 0
    assert abs(float(stats[1]["loss"]) - float(stats[0]["loss"])) <= 1e-4 * abs(float(stats[0]["loss"]))
    assert rel(stats[1]["new_logprobs"], stats[0]["new_logprobs"]) < 1e-4
    assert rel(grads[1], grads[0]) < 1e-4
    last = torch.linspace(0.2, 0.9, P, device="cuda")
    sq, sr = shape_rollout(q, last, relative=model.relative), shape_rollout(ref, last, relative=model.relative)
    assert rel(sq["kl"], sr["kl"]) < 1e-4 and rel(sq["scores"], sr["scores"]) < 1e-4


def test_every_prompt_in_flight_needs_no_refill(device_draws):
    model, emb, ref = device_draws
    q = model.sample_rollouts(*emb, slots=P, max_inference_steps=T_MAX, generator=torch.Generator().manual_seed(7))
    _assert_same_rollouts(q, ref)
    T = ref.sigmas.shape[1]
    assert q.device_steps <= T + 1                              # the longest trajectory + the look-ahead step
    assert ref.prob_masks.numel() == P * T and int(q.steps.sum()) < P * T   # the lockstep batch ran P x T slot-steps


def test_rloo_update_through_the_queue_end_to_end_tiny():
    """test_rloo_update_end_to_end_tiny with the rollouts drained through 3 queue slots."""
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModelRLOOWrapper
    from tpdm_b200.rloo import rloo_update
    from tpdm_b200.tpm_training import TimePredictorTrainer

    torch.manual_seed(3)
    tcfg = dict(sample_size=32, num_layers=2, attention_head_dim=96, num_attention_heads=4, caption_projection_dim=384, pos_embed_max_size=96)
    w = SD3PredictNextTimeStepModelRLOOWrapper(transformer_config=tcfg, torch_dtype=torch.float32, device="cuda", min_sigma=0.01,
                                               max_inference_steps=6)
    g = torch.Generator().manual_seed(0)
    data = dict(prompt=["a", "b"], prompt_embeds=torch.randn(2, 333, 4096, generator=g).cuda(),
                negative_prompt_embeds=torch.randn(2, 333, 4096, generator=g).cuda(),
                pooled_prompt_embeds=torch.randn(2, 2048, generator=g).cuda(),
                negative_pooled_prompt_embeds=torch.randn(2, 2048, generator=g).cuda())
    trainer = TimePredictorTrainer(w.agent_model.time_predictor, grid=16, max_samples=4 * 6, lr=1e-3)
    before = {k: v.clone() for k, v in w.agent_model.time_predictor.state_dict().items()}
    t_before = w.agent_model.transformer.proj_out.weight.clone()
    res = rloo_update(w, trainer, data, reward_fn=lambda lat, out: -(lat.float() ** 2).mean(dim=(1, 2, 3)), rloo_k=2, num_ppo_epochs=2,
                      micro_batch_size=2, slots=3)
    assert len(res["logs"]) == 4 and all(torch.isfinite(torch.tensor(l["loss"])) for l in res["logs"])
    assert abs(float(res["advantages"].reshape(2, -1).sum(0).abs().max())) < 1e-5
    assert abs(res["logs"][0]["ratio"] - 1.0) < 5e-3                                      # first replay reproduces the rollout log-probs
    after = w.agent_model.time_predictor.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert torch.equal(t_before, w.agent_model.transformer.proj_out.weight)


def test_argument_errors(device_draws):
    from tpdm_b200 import _lib as L

    model, emb, _ = device_draws
    eng = model.get_engine()
    lat = torch.randn(P, 16, 32, 32, device="cuda")
    with pytest.raises(ValueError):
        eng.sample_queue(lat, *emb, SLOTS, T_MAX, 7.0, schedule="lpt", predict=False)
    with pytest.raises(ValueError):
        model.sample_rollouts(*emb, latents=lat, slots=SLOTS, max_inference_steps=T_MAX, ratios=torch.full((P, T_MAX - 1), 0.7, device="cuda"))
    for slots in (0, P + 1):
        with pytest.raises(ValueError):
            model.sample_rollouts(*emb, latents=lat, slots=slots, max_inference_steps=T_MAX)
    plan = eng.plan(1, True, 32, 333, 3)          # a plan no queue has begun on
    with pytest.raises(RuntimeError):
        L.check(L.load().tpdm_queue_set_rollout(plan.handle, 0, None, None, None, None, None, None))
