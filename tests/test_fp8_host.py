"""CPU checks of the opt-in FP8 (E4M3) mode: the tests' fake quantization (fp8_fake_quant.py) (the rounding tpdm_quantize_fp8_rows implements) and
the validation of ``mmdit_precision``."""
import pytest
import torch


def _e4m3_table():
    """All finite E4M3 values (codes 0x00-0x7e and 0x80-0xfe) with their codes."""
    codes = torch.tensor([c for c in range(256) if (c & 0x7F) != 0x7F], dtype=torch.uint8)
    return codes.view(torch.float8_e4m3fn).float(), codes


def _nearest_even_e4m3(y: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even onto the E4M3 grid by brute force (|y| <= 448): the code whose value is nearest; on a tie the
    one with an even mantissa (even code)."""
    vals, codes = _e4m3_table()
    d = (y.reshape(-1, 1).double() - vals.double().reshape(1, -1)).abs()
    best = d.min(dim=1, keepdim=True).values
    cand = (d == best) & ((codes.reshape(1, -1) & 1) == 0)
    tie_free = (d == best).sum(1) == 1
    pick = torch.where(tie_free, (d == best).int().argmax(1), cand.int().argmax(1))
    out = codes[pick].reshape(y.shape)
    # +0 / -0: the sign of zero follows the input
    neg0 = (vals[pick] == 0).reshape(y.shape) & (torch.signbit(y))
    return torch.where(neg0, torch.full_like(out, 0x80), torch.where(vals[pick].reshape(y.shape) == 0, torch.zeros_like(out), out))


def test_fake_quant_codes_are_round_to_nearest_even_e4m3():
    from fp8_fake_quant import quantize_e4m3_rows

    g = torch.Generator().manual_seed(0)
    x = torch.randn(16, 384, generator=g) * torch.logspace(-3, 2, 16).reshape(-1, 1)
    codes, scale = quantize_e4m3_rows(x)
    assert codes.dtype == torch.float8_e4m3fn and scale.dtype == torch.float32 and scale.shape == (16,)
    amax = x.abs().amax(1)
    assert torch.equal(scale, amax / 448.0)
    y = x * (448.0 / amax).reshape(-1, 1)
    assert torch.equal(codes.view(torch.uint8), _nearest_even_e4m3(y))
    # every row's largest entry lands exactly on +-448
    top = codes.float().abs().amax(1)
    assert torch.equal(top, torch.full((16,), 448.0))


def test_zero_and_outlier_rows():
    from fp8_fake_quant import fake_quant_e4m3_rows, quantize_e4m3_rows

    x = torch.zeros(3, 128)
    x[1, 5] = 1000.0                                  # one outlier over tiny values: they fall onto E4M3 subnormals / zero
    x[1, 6:] = torch.linspace(-0.5, 0.5, 122)
    x[2] = torch.linspace(-1e-30, 1e-30, 128)          # tiny but normal fp32 magnitudes: the scale absorbs them
    codes, scale = quantize_e4m3_rows(x)
    assert float(scale[0]) == 1.0 and int(codes[0].view(torch.uint8).abs().sum()) == 0
    assert float(scale[1]) == float(torch.tensor(1000.0) / 448.0) and float(codes[1, 5].float()) == 448.0
    sub = codes[1, 6:].float().abs()
    assert float(sub.max()) <= 0.5 * 448.0 / 1000.0 + 1e-3 and bool((sub < 2 ** -6).any())   # subnormal E4M3 codes present
    assert float(codes[2].float().abs().max()) == 448.0
    fq = fake_quant_e4m3_rows(x)
    assert torch.equal(fq[0], x[0])
    assert float((fq[2] - x[2]).abs().max()) <= 1e-30 * 2 ** -3      # 3 mantissa bits at the row's own scale


def test_set_fp8_fake_quant_keeps_state_dict_and_switches_back():
    from fp8_fake_quant import FakeQuantE4M3Linear, set_fp8_fake_quant
    from oracle import sd3_oracle as O

    torch.manual_seed(0)
    m = O.OracleSD3Transformer(O.tiny_config()).eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    inp = O.synthetic_inputs(O.tiny_config(), batch=1)
    args = (inp["latents"], inp["prompt_embeds"], inp["pooled_prompt_embeds"], torch.tensor([500.0]))
    with torch.no_grad():
        ref = m(*args)[0]
        set_fp8_fake_quant(m)
        fq = m(*args)[0]
        assert sd.keys() == m.state_dict().keys()
        assert isinstance(m.transformer_blocks[0].attn.add_q_proj, FakeQuantE4M3Linear)
        assert not isinstance(m.transformer_blocks[0].attn.to_out[0], FakeQuantE4M3Linear)
        assert not isinstance(m.transformer_blocks[0].ff.net[2], FakeQuantE4M3Linear)
        set_fp8_fake_quant(m, False)
        back = m(*args)[0]
    assert torch.equal(back, ref)
    err = float((fq - ref).norm() / ref.norm())
    assert 1e-4 < err < 1e-1, err


def test_mmdit_precision_validation():
    from tpdm_b200.engine import Engine
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel, SD3PredictNextTimeStepModelRLOOWrapper
    from tpdm_b200.transformer_sd3 import CustomSD3Transformer2DModel

    tcfg = dict(sample_size=32, num_layers=2, attention_head_dim=96, num_attention_heads=4, caption_projection_dim=384, pos_embed_max_size=96)
    t = CustomSD3Transformer2DModel(**tcfg)
    assert t.mmdit_precision == "bf16"
    t.mmdit_precision = "fp8"
    assert t.mmdit_precision == "fp8"
    with pytest.raises(ValueError):
        t.mmdit_precision = "fp16"
    assert t.mmdit_precision == "fp8"
    with pytest.raises(ValueError):
        CustomSD3Transformer2DModel(**tcfg, mmdit_precision="e4m3")
    m = SD3PredictNextTimeStepModel(transformer_config=tcfg, torch_dtype=torch.float32, mmdit_precision="fp8")
    assert m.mmdit_precision == "fp8" and m.transformer.mmdit_precision == "fp8"
    m.mmdit_precision = "bf16"
    assert m.transformer.mmdit_precision == "bf16"
    with pytest.raises(ValueError):
        SD3PredictNextTimeStepModel(transformer_config=tcfg, torch_dtype=torch.float32, mmdit_precision="int8")
    w = SD3PredictNextTimeStepModelRLOOWrapper(transformer_config=tcfg, torch_dtype=torch.float32, mmdit_precision="fp8")
    assert w.agent_model.transformer.mmdit_precision == "fp8"
    with pytest.raises(ValueError):      # validated before the library or a device is touched
        Engine({}, torch.device("cpu"), mmdit_precision="FP8")


def test_build_fp8_gemm_uses_utcqmma_without_spills():
    """The CTA-pair GEMM object that build() leaves: the E4M3 instantiation issues UTCQMMA (kind::f8f6f4), the bf16 one UTCHMMA
    only, and ptxas reports no spills for either."""
    import os
    import re
    import shutil
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    obj = os.path.join(root, "tpdm_b200", "_build", "gemm2_tcgen05.o")
    log = obj.replace(".o", ".cu.log")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not (os.path.exists(obj) and os.path.exists(log) and os.path.exists(cuobjdump)):
        pytest.skip("the library has not been built here (python -m tpdm_b200.build) or cuobjdump is missing")
    text = open(log).read()
    entries = re.findall(r"Compiling entry function '(\w*gemm2_bf16_tcgen05_kernel\w*)'.*?\n.*?\n(.*?)\n", text)
    assert len(entries) == 2, entries
    for _, info in entries:
        assert "0 bytes spill stores, 0 bytes spill loads" in info, info
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs = dict(re.findall(r"Function : (\S+)\n(.*?)(?=\n\s+Function : |\Z)", sass, flags=re.S))
    fp8 = [b for n, b in funcs.items() if "gemm2_bf16_tcgen05_kernelILb1E" in n]
    bf16 = [b for n, b in funcs.items() if "gemm2_bf16_tcgen05_kernelILb0E" in n]
    assert len(fp8) == 1 and len(bf16) == 1
    assert "UTCQMMA" in fp8[0] and "UTCHMMA" not in fp8[0]
    assert "UTCHMMA" in bf16[0] and "UTCQMMA" not in bf16[0]
    assert "STL" not in fp8[0] and "LDL" not in fp8[0]
