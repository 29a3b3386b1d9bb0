"""Open prompt stream (tpdm_stream_*, Engine.open_stream, SD3PredictNextTimeStepModel.open_prompt_stream): prompts admitted
into a running device-side queue, results collected as each request finishes.  Every request must give what batch-1
``forward(predict=True)`` gives it, with the bars of the closed-queue test (same step count, sigmas within 1e-5, final latent
rel-L2 < 1e-4)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

TINY = dict(sample_size=32, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=96, num_attention_heads=4, joint_attention_dim=4096,
            caption_projection_dim=384, pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=96)
P, T = 9, 12


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def tiny_model(precision="bf16"):
    """The closed-queue test's model: the TimePredictor is made input-sensitive so that trajectory lengths differ."""
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    torch.manual_seed(21)
    model = SD3PredictNextTimeStepModel(transformer_config=TINY, torch_dtype=torch.float32, device="cuda", min_sigma=0.05,
                                        mmdit_precision=precision)
    with torch.no_grad():
        tp = model.time_predictor
        tp.fc2.weight.mul_(40)
        tp.fc1.weight.mul_(8)
        tp.conv2.weight.mul_(6)
        tp.norm1.linear.weight.mul_(4)
    return model


def make_inputs():
    """The closed-queue test's 7 prompts (their trajectory lengths differ), plus prompts 1 and 4 again with other noise scales."""
    g = torch.Generator().manual_seed(3)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    pe, ne, pp, npp, lat = mk(7, 333, 4096), mk(7, 333, 4096), mk(7, 2048), mk(7, 2048), mk(7, 16, 32, 32)
    lat = lat * torch.linspace(0.5, 2.0, 7, device="cuda").view(7, 1, 1, 1)
    extra = [1, 4]
    cat = lambda t, x=None: torch.cat([t, t[extra] if x is None else t[extra] * x])
    return dict(prompt_embeds=cat(pe), negative_prompt_embeds=cat(ne), pooled_prompt_embeds=cat(pp), negative_pooled_prompt_embeds=cat(npp),
                latents=cat(lat, 1.3))


def per_prompt(model, inp):
    ref = []
    for i in range(P):
        o = model(**{k: v[i:i + 1] for k, v in inp.items()}, max_inference_steps=T, predict=True)
        ref.append((o.sigmas.shape[1], o.sigmas[0], o.latents[0]))
    return ref


@pytest.fixture(scope="module")
def tiny():
    model = tiny_model()
    inp = make_inputs()
    ref = per_prompt(model, inp)
    assert len({r[0] for r in ref}) > 1, [r[0] for r in ref]     # the stress is real: lengths differ
    return model, inp, ref


def sub(s, inp, lo, hi):
    return s.submit(**{k: v[lo:hi] for k, v in inp.items()})


def check(res, ref, prompt_of):
    assert len(res) == len(prompt_of)
    for rid, r in res.items():
        n, sig, lat = ref[prompt_of[rid]]
        assert r["steps"] == n, (rid, r["steps"], n)
        assert r["sigmas"].shape == (n,) and torch.allclose(r["sigmas"], sig, atol=1e-5)
        assert rel(r["latents"], lat) < 1e-4


def scripted(model, inp, use_graph):
    """3 prompts, two steps, admissions as entries free up (a submit that only partly fits raises and admits nothing), a fully
    idle stream, then the last two prompts."""
    res, prompt_of = {}, {}
    with model.open_prompt_stream(slots=3, capacity=4, max_inference_steps=T, use_graph=use_graph) as s:
        for i, rid in enumerate(sub(s, inp, 0, 3)):
            prompt_of[rid] = i
        s.step()
        s.step()
        with pytest.raises(RuntimeError):
            sub(s, inp, 3, 5)                 # one entry is free
        nxt = 3
        while nxt < 7:
            s.step()
            res.update(s.results())
            free = 4 - (nxt - len(res))
            if free > 0:
                k = min(free, 7 - nxt)
                for j, rid in enumerate(sub(s, inp, nxt, nxt + k)):
                    prompt_of[rid] = nxt + j
                nxt += k
        res.update(s.drain())
        assert len(res) == 7 and sorted(res) == list(range(7))     # request ids are handed out in submission order
        d0 = s.device_steps
        s.step(3)                             # idle and fully harvested: nothing runs
        assert s.device_steps == d0 and s.results() == {}
        for j, rid in enumerate(sub(s, inp, 7, 9)):
            prompt_of[rid] = 7 + j
        res.update(s.drain())
        steps = s.device_steps
    return res, prompt_of, steps


def test_scripted_admissions_match_forward_and_graph_replay(tiny):
    model, inp, ref = tiny
    res, prompt_of, steps = scripted(model, inp, use_graph=True)
    check(res, ref, prompt_of)
    assert steps < sum(r[0] for r in ref)
    eager, prompt_of_e, steps_e = scripted(model, inp, use_graph=False)
    assert prompt_of_e == prompt_of and steps_e == steps
    for rid in res:
        assert eager[rid]["steps"] == res[rid]["steps"] and rel(eager[rid]["latents"], res[rid]["latents"]) < 1e-6


def test_idle_stream_runs_nothing_and_starts_a_new_request_at_once(tiny):
    model, inp, ref = tiny
    with model.open_prompt_stream(slots=2, capacity=2, max_inference_steps=T) as s:
        s.step(4)
        assert s.device_steps == 0 and s.results() == {}
        for i in (4, 1):
            d0 = s.device_steps
            (rid,) = sub(s, inp, i, i + 1)
            res = s.drain()
            check(res, ref, {rid: i})
            assert s.device_steps - d0 <= ref[i][0] + 1
            s.step(2)
            assert s.device_steps - d0 <= ref[i][0] + 1


def test_forward_and_sample_queue_between_stream_steps(tiny):
    model, inp, ref = tiny
    res, prompt_of = {}, {}
    with model.open_prompt_stream(slots=3, capacity=5, max_inference_steps=T) as s:
        for j, rid in enumerate(sub(s, inp, 2, 7)):
            prompt_of[rid] = 2 + j
        s.step(2)
        o = model(**{k: v[0:1] for k, v in inp.items()}, max_inference_steps=T, predict=True)
        s.step()
        q = model.sample_queue(inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["pooled_prompt_embeds"],
                               inp["negative_pooled_prompt_embeds"], latents=inp["latents"], slots=3, max_inference_steps=T)
        res.update(s.results())
        res.update(s.drain())
    check(res, ref, prompt_of)
    assert o.sigmas.shape[1] == ref[0][0] and rel(o.latents[0], ref[0][2]) < 1e-4
    assert q.steps.tolist() == [r[0] for r in ref]
    for i in range(P):
        assert rel(q.latents[i], ref[i][2]) < 1e-4


def test_fp8_stream_matches_fp8_forward():
    model = tiny_model("fp8")
    inp = make_inputs()
    ref = per_prompt(model, inp)
    res, prompt_of = {}, {}
    with model.open_prompt_stream(slots=3, capacity=P, max_inference_steps=T) as s:
        for j, rid in enumerate(sub(s, inp, 0, P)):
            prompt_of[rid] = j
        res.update(s.drain())
    check(res, ref, prompt_of)


def test_time_predictor_refresh_waits_for_the_stream(tiny):
    """get_engine refreshes the packed TimePredictor after its weights change: refused while stream requests are in flight (they
    would switch weights mid-trajectory), allowed once they are collected."""
    model, inp, ref = tiny
    with model.open_prompt_stream(slots=2, capacity=2, max_inference_steps=T) as s:
        (rid,) = sub(s, inp, 3, 4)
        s.step()
        with torch.no_grad():
            model.time_predictor.fc1.bias.mul_(1.0)      # same values, new version: the engine must re-pack
        with pytest.raises(RuntimeError):
            model(**{k: v[0:1] for k, v in inp.items()}, max_inference_steps=T, predict=True)
        check(s.drain(), ref, {rid: 3})
        o = model(**{k: v[0:1] for k, v in inp.items()}, max_inference_steps=T, predict=True)
        assert o.sigmas.shape[1] == ref[0][0] and rel(o.latents[0], ref[0][2]) < 1e-4
        (rid,) = sub(s, inp, 5, 6)
        check(s.drain(), ref, {rid: 5})


def test_stream_errors(tiny):
    from tpdm_b200 import _lib as L

    model, inp, _ = tiny
    s = model.open_prompt_stream(slots=2, capacity=3, max_inference_steps=T)
    bad = dict((k, v[0:1]) for k, v in inp.items())
    with pytest.raises(ValueError):
        s.submit(**dict(bad, prompt_embeds=inp["prompt_embeds"][0:1, :300]))          # text length other than the plan's
    with pytest.raises(ValueError):
        s.submit(**dict(bad, latents=inp["latents"][0:1, :, :16, :16]))
    with pytest.raises(ValueError):
        s.submit(**dict(bad, pooled_prompt_embeds=inp["pooled_prompt_embeds"][0:2]))
    sub(s, inp, 0, 3)
    with pytest.raises(RuntimeError):
        sub(s, inp, 3, 4)                     # the ring is full
    lib = L.load()
    dummy = torch.zeros(1024, device="cuda")
    d = L.ptr(dummy)
    st = lib.tpdm_queue_begin(s._plan.handle, 3, d, d, d, d, d, 7.0, d, 1 << 20, d, d, d, None, None, 0, None, 0, None)
    assert st == L.TPDM_ERR_STATE and b"open prompt stream" in lib.tpdm_last_error()
    assert lib.tpdm_stream_open(s._plan.handle, 3, 7.0, d, 1 << 20, None) == L.TPDM_ERR_STATE
    # entry ids are checked before anything is enqueued: repeated ids, more prompts than entries, ids out of range
    assert lib.tpdm_stream_submit(s._plan.handle, 2, (C.c_int * 2)(1, 1), d, d, d, d, d, None) == L.TPDM_ERR_ARG
    assert b"twice" in lib.tpdm_last_error()
    assert lib.tpdm_stream_submit(s._plan.handle, 4, (C.c_int * 4)(0, 1, 2, 0), d, d, d, d, d, None) == L.TPDM_ERR_ARG
    assert lib.tpdm_stream_submit(s._plan.handle, 1, (C.c_int * 1)(3), d, d, d, d, d, None) == L.TPDM_ERR_ARG
    res = s.drain()
    assert len(res) == 3
    s.close()
    with pytest.raises(RuntimeError):
        sub(s, inp, 0, 1)
    assert lib.tpdm_stream_submit(s._plan.handle, 1, (C.c_int * 1)(0), d, d, d, d, d, None) == L.TPDM_ERR_STATE
    with pytest.raises(RuntimeError):
        s.step()


def test_sd3_medium_1024_stream_matches_closed_queue():
    """Full-size admission GEMM (K 4096, N 1536, 333 text rows per prompt) and steps: the first 8 prompts of
    ``bench.py --workload config3`` (same model seed, TimePredictor scaling and per-prompt inputs, 7-28 step trajectories), 2 slots,
    a ring of 3 entries refilled as requests finish; the closed queue over the same prompts gives the same steps and latents."""
    from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel

    torch.manual_seed(1234)
    model = SD3PredictNextTimeStepModel(transformer_config=dict(SD3_MEDIUM_TRANSFORMER_CONFIG), torch_dtype=torch.bfloat16, device="cuda",
                                        init_alpha=1.5, init_beta=0.5)
    with torch.no_grad():
        tp = model.time_predictor
        tp.fc2.weight.mul_(4.0)
        tp.fc1.weight.mul_(4.0)
        tp.conv2.weight.mul_(2.0)
    n, cap = 8, 3

    def prompt(i):
        g = torch.Generator().manual_seed(5000 + i)
        mk = lambda *s: torch.randn(*s, generator=g).cuda()
        return [mk(1, 333, 4096), mk(1, 333, 4096), mk(1, 2048), mk(1, 2048), mk(1, 16, 128, 128)]

    cols = list(zip(*[prompt(i) for i in range(n)]))
    inp = dict(zip(("prompt_embeds", "negative_prompt_embeds", "pooled_prompt_embeds", "negative_pooled_prompt_embeds", "latents"),
                   [torch.cat(c) for c in cols]))
    q = model.sample_queue(inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["pooled_prompt_embeds"], inp["negative_pooled_prompt_embeds"],
                           latents=inp["latents"], slots=2, max_inference_steps=28)
    assert len(set(q.steps.tolist())) > 1, q.steps.tolist()       # slots are refilled at different steps
    res, prompt_of = {}, {}
    with model.open_prompt_stream(slots=2, capacity=cap, max_inference_steps=28) as s:
        nxt = 0
        while nxt < n:
            free = cap - (nxt - len(res))
            if free > 0:
                k = min(free, n - nxt)
                for j, rid in enumerate(sub(s, inp, nxt, nxt + k)):
                    prompt_of[rid] = nxt + j
                nxt += k
            s.step()
            res.update(s.results())
        res.update(s.drain())
    assert len(res) == n
    for rid, r in res.items():
        i = prompt_of[rid]
        assert r["steps"] == int(q.steps[i])
        assert torch.allclose(r["sigmas"], q.sigmas[i, 1: r["steps"] + 1], atol=1e-5)
        assert rel(r["latents"], q.latents[i]) < 1e-4
