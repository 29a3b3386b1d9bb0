"""Per-request options of the open prompt stream: guidance scale, step cap and schedule mode (Beta mode, or Beta draws from the
request's own seed).  A request with options (g, m, predict, seed) must give what batch-1 ``forward(guidance_scale=g,
max_inference_steps=m, predict=...)`` gives it (for predict=False: with that Philox seed), with the bars of the stream tests:
equal step count, sigmas within 1e-5, final latent and alpha / beta / log-prob rel-L2 < 1e-4."""
import ctypes as C

import pytest
import torch

from test_prompt_stream_gpu import P, T, make_inputs, rel, tiny_model

GUIDANCE = [1.0, 2.0, 3.5, 5.0, 7.0, 9.0, 12.0, 4.0, 6.0]
REC = ("alphas", "betas", "logprobs")


def one(inp, i):
    return {k: v[i:i + 1] for k, v in inp.items()}


def forward_ref(model, inp, i, **kw):
    """(steps, sigmas, latents, alphas, betas, logprobs) of batch-1 forward of prompt i (``latents=None``: drawn from the
    generator)."""
    kw.setdefault("max_inference_steps", T)
    kw.setdefault("predict", True)
    o = model(**dict(one(inp, i), **kw))
    n = o.sigmas.shape[1]
    return dict(steps=n, sigmas=o.sigmas[0], latents=o.latents[0], alphas=o.alphas[0, :n], betas=o.betas[0, :n], logprobs=o.logprobs[0, :n])


def close(a, b):
    """rel-L2 < 1e-4 over the finite elements, the others equal: the tiny model's TimePredictor can overflow to beta = inf,
    whose log-prob is NaN in forward and in the stream alike."""
    fin = torch.isfinite(b)
    same = torch.isclose(a[~fin], b[~fin], rtol=0.0, atol=0.0, equal_nan=True).all()
    return torch.equal(torch.isfinite(a), fin) and bool(same) and rel(a[fin], b[fin]) < 1e-4


def check_one(r, ref):
    n = ref["steps"]
    assert r["steps"] == n, (r["steps"], n)
    assert r["sigmas"].shape == (n,) and torch.allclose(r["sigmas"], ref["sigmas"], atol=1e-5), (r["sigmas"], ref["sigmas"])
    assert rel(r["latents"], ref["latents"]) < 1e-4
    for k in REC:
        assert r[k].shape == (n,) and close(r[k], ref[k]), (k, r[k], ref[k])


def run_stream(model, submits, slots=3, capacity=P, use_graph=True, max_steps=T):
    """Submits each (lo, hi, inputs, options) in order, drains, and returns ({request id: result}, [request ids per submit],
    device steps)."""
    with model.open_prompt_stream(slots=slots, capacity=capacity, max_inference_steps=max_steps, use_graph=use_graph) as s:
        rids = [s.submit(**{k: v[lo:hi] for k, v in inp.items()}, **opts) for lo, hi, inp, opts in submits]
        res = s.drain()
        return res, rids, s.device_steps


def latents_and_seed(model, gen, n=1):
    """What forward(generator=gen) draws: the latents, then one Philox seed per prompt."""
    side = model.default_sample_size * model.vae_scale_factor
    lat = model.prepare_latents(n, model.transformer.config.in_channels, side, side, torch.float32, model.device, gen)
    seeds = torch.randint(0, 2**62, (n,), generator=gen).tolist()
    return lat, seeds


@pytest.fixture(scope="module")
def tiny():
    return tiny_model(), make_inputs()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp8"])
def test_mixed_guidance_matches_forward(precision, tiny):
    model, inp = tiny if precision == "bf16" else (tiny_model(precision), tiny[1])
    refs = [forward_ref(model, inp, i, guidance_scale=g) for i, g in enumerate(GUIDANCE)]
    res, (rids,), _ = run_stream(model, [(0, P, inp, dict(guidance_scale=GUIDANCE))])
    assert len(res) == P
    for i, rid in enumerate(rids):
        check_one(res[rid], refs[i])
    # not vacuous: the guidance reaches the trajectory
    assert rel(forward_ref(model, inp, 0, guidance_scale=7.0)["latents"], refs[0]["latents"]) > 1e-2


@pytest.mark.gpu
def test_step_caps_match_forward_and_bad_caps_admit_nothing(tiny):
    model, inp = tiny
    caps = [(2, 4, T)[i % 3] for i in range(P)]
    refs = [forward_ref(model, inp, i, max_inference_steps=m) for i, m in enumerate(caps)]
    assert any(r["steps"] == m and float(r["sigmas"][-1]) >= model.min_sigma for r, m in zip(refs, caps))   # stopped by its cap
    res, (rids,), _ = run_stream(model, [(0, P, inp, dict(max_inference_steps=caps))])
    for i, rid in enumerate(rids):
        check_one(res[rid], refs[i])
    with model.open_prompt_stream(slots=2, capacity=3, max_inference_steps=T) as s:
        x = {k: v[0:2] for k, v in inp.items()}
        for bad in (dict(max_inference_steps=T + 1), dict(max_inference_steps=0), dict(max_inference_steps=[4, T + 1]),
                    dict(max_inference_steps=[4]), dict(guidance_scale=float("nan")), dict(guidance_scale=[7.0, float("inf")]),
                    dict(predict=False, seed=-1), dict(predict=False, seed=2**64), dict(seed=[1, 2, 3])):
            with pytest.raises(ValueError):
                s.submit(**x, **bad)
        torch.cuda.synchronize()
        assert s._counters[:3].tolist() == [0, 0, 0] and len(s._free) == 3 and s.device_steps == 0
        (rid, _) = s.submit(**x, max_inference_steps=2)
        assert s.drain()[rid]["steps"] <= 2


@pytest.mark.gpu
def test_sampled_requests_match_forward(tiny):
    model, inp = tiny
    sampled = [0, 2, 3, 5]
    lat, seeds, refs = [], [], []
    for i in range(6):
        if i in sampled:
            refs.append(forward_ref(model, inp, i, predict=False, generator=torch.Generator().manual_seed(100 + i), latents=None))
            la, (sd,) = latents_and_seed(model, torch.Generator().manual_seed(100 + i))
            lat.append(la)
            seeds.append(sd)
        else:
            refs.append(forward_ref(model, inp, i))
            lat.append(inp["latents"][i:i + 1])
            seeds.append(0)
    x = dict({k: v[:6] for k, v in inp.items()}, latents=torch.cat(lat))
    opts = dict(predict=[i not in sampled for i in range(6)], seed=seeds)
    res, (rids,), _ = run_stream(model, [(0, 6, x, opts)])
    for i, rid in enumerate(rids):
        check_one(res[rid], refs[i])
    # every prompt with seed 11, 11 again and 12: the same seed gives the same result, another seed other schedules (some
    # prompts end at their first step whatever the draw, so at least one prompt must differ)
    y = {k: torch.cat([v] * 3) for k, v in inp.items()}
    res, (rids,), _ = run_stream(model, [(0, 3 * P, y, dict(predict=False, seed=[11] * (2 * P) + [12] * P))], capacity=3 * P)
    a, b, c = ([res[r] for r in rids[j * P:(j + 1) * P]] for j in range(3))
    for x, z in zip(a, b):
        assert x["steps"] == z["steps"] and torch.equal(x["sigmas"], z["sigmas"]) and torch.equal(x["latents"], z["latents"])
    assert any(x["steps"] != z["steps"] or not torch.allclose(x["sigmas"], z["sigmas"], atol=1e-3) for x, z in zip(a, c))


@pytest.mark.gpu
def test_generator_form_equals_explicit_seeds(tiny):
    model, inp = tiny
    emb = {k: v[:4] for k, v in inp.items() if k != "latents"}
    with model.open_prompt_stream(slots=2, capacity=4, max_inference_steps=T) as s:
        rids = s.submit(**emb, generator=torch.Generator().manual_seed(9), predict=False)
        got = s.drain()
    lat, seeds = latents_and_seed(model, torch.Generator().manual_seed(9), 4)
    assert len(set(seeds)) == 4
    res, (rids_e,), _ = run_stream(model, [(0, 4, dict(emb, latents=lat), dict(predict=False, seed=seeds))], slots=2, capacity=4)
    for r, e in zip(rids, rids_e):
        assert got[r]["steps"] == res[e]["steps"]
        for k in ("latents", "sigmas") + REC:
            assert torch.equal(got[r][k], res[e][k]), k


def mixed_script(model, inp, use_graph):
    """Guidance, caps and sampled requests mixed in three slots, admitted in two submissions."""
    first = dict(guidance_scale=[3.5, 7.0, 9.0, 5.0], max_inference_steps=[T, 4, T, 2], predict=[True, False, True, False],
                 seed=[0, 21, 0, 22])
    second = dict(guidance_scale=[12.0, 2.0, 7.0, 1.0, 5.0], max_inference_steps=[T, T, 3, T, T], predict=[False, True, True, False, True],
                  seed=[23, 0, 0, 24, 0])
    return run_stream(model, [(0, 4, inp, first), (4, P, inp, second)], use_graph=use_graph)


@pytest.mark.gpu
def test_mixed_options_graph_and_eager_agree(tiny):
    model, inp = tiny
    g, rids_g, steps_g = mixed_script(model, inp, True)
    e, rids_e, steps_e = mixed_script(model, inp, False)
    assert rids_g == rids_e and steps_g == steps_e and len(g) == P
    for rid in g:
        assert g[rid]["steps"] == e[rid]["steps"]
        for k in ("latents", "sigmas") + REC:
            assert rel(g[rid][k], e[rid][k]) < 1e-6, (rid, k)
    # and each is its batch-1 forward, e.g. prompt 6 (guidance 7, cap 3)
    check_one(g[rids_g[1][2]], forward_ref(model, inp, 6, guidance_scale=7.0, max_inference_steps=3))


@pytest.mark.gpu
def test_lockstep_graph_follows_a_guidance_change(tiny, monkeypatch):
    model, inp = tiny
    x = one(inp, 2)
    model(**x, max_inference_steps=T, predict=True, guidance_scale=7.0)
    graph = model(**x, max_inference_steps=T, predict=True, guidance_scale=3.5)
    monkeypatch.setenv("TPDM_SAMPLE_GRAPH", "0")
    eager = model(**x, max_inference_steps=T, predict=True, guidance_scale=3.5)
    assert graph.sigmas.shape == eager.sigmas.shape and torch.allclose(graph.sigmas, eager.sigmas, atol=1e-6)
    assert rel(graph.latents, eager.latents) < 1e-6


def test_request_options_struct_is_24_bytes():
    from tpdm_b200 import _lib as L

    assert C.sizeof(L.TpdmRequestOptions) == 24
    assert [f[0] for f in L.TpdmRequestOptions._fields_] == ["guidance_scale", "max_steps", "predict", "reserved", "seed"]
    assert L.TpdmRequestOptions.seed.offset == 16


def raw_submit(s, inp, lo, hi, with_options):
    """PromptStream.submit's bookkeeping around a direct tpdm_stream_submit (or _options with NULL options) call."""
    from tpdm_b200 import _lib as L

    lib, n = L.load(), hi - lo
    ts = [inp[k][lo:hi].contiguous() for k in ("latents", "negative_prompt_embeds", "prompt_embeds", "negative_pooled_prompt_embeds",
                                                "pooled_prompt_embeds")]
    entries = s._free[len(s._free) - n:][::-1]
    ids = (C.c_int * n)(*entries)
    s._cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s._cs):
        ptrs = [L.ptr(t) for t in ts]
        if with_options:
            L.check(lib.tpdm_stream_submit_options(s._plan.handle, n, ids, *ptrs, None, L.stream_ptr()))
        else:
            L.check(lib.tpdm_stream_submit(s._plan.handle, n, ids, *ptrs, L.stream_ptr()))
    s._cs.synchronize()
    del s._free[len(s._free) - n:]
    rids = list(range(s._next_id, s._next_id + n))
    s._entry_req.update(zip(entries, rids))
    s._next_id += n
    s._submitted += n
    return rids


@pytest.mark.gpu
def test_c_abi_null_options_invalid_options_and_records(tiny):
    from tpdm_b200 import _lib as L

    model, inp = tiny
    lib = L.load()
    out = []
    for with_options in (False, True):
        with model.open_prompt_stream(slots=3, capacity=5, max_inference_steps=T, guidance_scale=5.0) as s:
            rids = raw_submit(s, inp, 2, 7, with_options)
            res = s.drain()
            out.append([res[r] for r in rids])
    for a, b in zip(*out):
        assert a["steps"] == b["steps"]
        for k in ("latents", "sigmas") + REC:
            assert torch.equal(a[k], b[k]), k
    check_one(out[1][0], forward_ref(model, inp, 2, guidance_scale=5.0))
    s = model.open_prompt_stream(slots=2, capacity=3, max_inference_steps=T)
    torch.cuda.synchronize()
    before = s._counters.tolist()
    d = L.ptr(torch.zeros(1024, device="cuda"))
    good = dict(guidance_scale=7.0, max_steps=T, predict=1, reserved=0, seed=0)
    for bad, word in ((dict(guidance_scale=float("nan")), b"finite"), (dict(guidance_scale=float("-inf")), b"finite"),
                      (dict(max_steps=0), b"max_steps"), (dict(max_steps=T + 1), b"max_steps"), (dict(predict=2), b"predict"),
                      (dict(predict=-1), b"predict"), (dict(reserved=1), b"reserved")):
        opts = (L.TpdmRequestOptions * 2)(L.TpdmRequestOptions(**good), L.TpdmRequestOptions(**dict(good, **bad)))
        st = lib.tpdm_stream_submit_options(s._plan.handle, 2, (C.c_int * 2)(0, 1), d, d, d, d, d, opts, None)
        assert st == L.TPDM_ERR_ARG and word in lib.tpdm_last_error(), (bad, lib.tpdm_last_error())
    torch.cuda.synchronize()
    assert s._counters.tolist() == before and before[:4] == [0] * 4
    ptrs = [L.vp() for _ in range(3)]
    assert lib.tpdm_stream_records(s._plan.handle, *[C.byref(p) for p in ptrs]) == 0 and all(p.value for p in ptrs)
    s.close()
    assert lib.tpdm_stream_records(s._plan.handle, *[C.byref(p) for p in ptrs]) == L.TPDM_ERR_STATE


@pytest.mark.gpu
def test_sd3_medium_1024_mixed_options_match_forward():
    """SD3-medium 1024^2 with the model seed, TimePredictor scaling and per-prompt inputs of
    test_sd3_medium_1024_stream_matches_closed_queue: 6 requests through 2 slots, guidance 3.5 or 7, one cap of 10, two sampled."""
    from tpdm_b200.modeling_sd3_pnt import SD3_MEDIUM_TRANSFORMER_CONFIG, SD3PredictNextTimeStepModel

    torch.manual_seed(1234)
    model = SD3PredictNextTimeStepModel(transformer_config=dict(SD3_MEDIUM_TRANSFORMER_CONFIG), torch_dtype=torch.bfloat16, device="cuda",
                                        init_alpha=1.5, init_beta=0.5)
    with torch.no_grad():
        tp = model.time_predictor
        tp.fc2.weight.mul_(4.0)
        tp.fc1.weight.mul_(4.0)
        tp.conv2.weight.mul_(2.0)
    n = 6

    def prompt(i):
        g = torch.Generator().manual_seed(5000 + i)
        mk = lambda *s: torch.randn(*s, generator=g).cuda()
        return [mk(1, 333, 4096), mk(1, 333, 4096), mk(1, 2048), mk(1, 2048), mk(1, 16, 128, 128)]

    cols = list(zip(*[prompt(i) for i in range(n)]))
    inp = dict(zip(("prompt_embeds", "negative_prompt_embeds", "pooled_prompt_embeds", "negative_pooled_prompt_embeds", "latents"),
                   [torch.cat(c) for c in cols]))
    guidance = [3.5, 7.0, 3.5, 7.0, 7.0, 3.5]
    caps = [28, 28, 28, 28, 10, 28]     # prompt 4 runs 28 steps uncapped (profiles/prompt_stream_n1.json)
    predict = [True, True, True, False, True, False]
    # forward draws its seed from Generator(100 + i) (the latents are given), the stream gets that draw
    seeds = [torch.randint(0, 2**62, (1,), generator=torch.Generator().manual_seed(100 + i)).item() if not predict[i] else 0 for i in range(n)]
    refs = []
    for i in range(n):
        gen = torch.Generator().manual_seed(100 + i)
        refs.append(forward_ref(model, inp, i, guidance_scale=guidance[i], max_inference_steps=caps[i], predict=predict[i], generator=gen))
    assert refs[4]["steps"] == 10 and float(refs[4]["sigmas"][-1]) >= model.min_sigma     # the cap ended it
    res, (rids,), _ = run_stream(model, [(0, n, inp, dict(guidance_scale=guidance, max_inference_steps=caps, predict=predict, seed=seeds))],
                                 slots=2, capacity=n, max_steps=28)
    for i, rid in enumerate(rids):
        check_one(res[rid], refs[i])
