"""CPU tests of the oracle (-m "not gpu"): the restatement must reproduce the golden vectors that
tests/golden/make_golden.py recorded from the UNMODIFIED reference modules."""
import json
import os

import pytest
import torch
from safetensors.torch import load_file

from oracle import cases, dit_oracle, vae_oracle

FAST_DIT = ["tiny_t2", "tiny_t8", "tiny_b2", "tiny_ragged"]
FAST_VAE = ["tiny_5f", "tiny_9f", "tiny_1f"]


def _manifest(golden_dir):
    with open(os.path.join(golden_dir, "MANIFEST.json")) as f:
        return json.load(f)["cases"]


@pytest.mark.parametrize("name", FAST_DIT)
def test_dit_oracle_matches_golden(name, golden_dir):
    case = cases.DIT_CASES[name]
    gold = load_file(os.path.join(golden_dir, f"dit_{name}.safetensors"))
    man = _manifest(golden_dir)[f"dit_{name}"]
    sd = cases.dit_weights(case)
    x, t, text, img = cases.dit_inputs(case)
    wsum = cases.checksum(torch.cat([v.flatten()[:4096].float() for v in sd.values()]))
    assert abs(wsum - man["weights_checksum"]) <= 1e-9 * abs(man["weights_checksum"]), "seeded weights drifted"
    with torch.no_grad():
        out, inter = dit_oracle.dit_forward(sd, case.cfg, x, t, text, img, return_intermediates=True)
    torch.testing.assert_close(out, gold["out_fp32"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(inter["timestep_proj"], gold["timestep_proj_fp32"], rtol=1e-5, atol=1e-6)
    if "block0_fp32" in gold:
        torch.testing.assert_close(inter["block0"], gold["block0_fp32"], rtol=1e-5, atol=1e-6)
    # bf16 configuration of the CLI (run_inference_diffusers.py:341-353)
    sdb = cases.to_bf16_state(sd)
    with torch.no_grad():
        outb = dit_oracle.dit_forward(sdb, case.cfg, x.bfloat16(), t, text.bfloat16(), img.bfloat16())
    assert outb.dtype == torch.bfloat16
    # same CPU kernels as at generation time -> bit-exact; tolerate 1 bf16 ulp should a BLAS path differ between hosts
    diff = (outb.float() - gold["out_bf16"].float()).abs()
    assert diff.max() <= 2.0 * man["bf16_vs_fp32_maxabs"]
    assert diff.mean() <= 0.25 * man["bf16_vs_fp32_meanabs"] + 1e-9


@pytest.mark.parametrize("name", FAST_VAE)
def test_vae_oracle_matches_golden(name, golden_dir):
    case = cases.VAE_CASES[name]
    gold = load_file(os.path.join(golden_dir, f"vae_{name}.safetensors"))
    sd = cases.vae_weights(case)
    video, z = cases.vae_inputs(case)
    mu = vae_oracle.vae_encode(sd, case.cfg, video)
    dec = vae_oracle.vae_decode(sd, case.cfg, z, clamp=False)
    torch.testing.assert_close(mu, gold["mu_fp32"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(dec, gold["dec_fp32"], rtol=1e-4, atol=1e-5)
    assert mu.shape == (1, 16, 1 + (case.frames_px - 1) // 4, case.height // 8, case.width // 8)
    assert dec.shape == (1, 3, case.frames_px, case.height, case.width)
    assert vae_oracle.vae_decode(sd, case.cfg, z).abs().max() <= 1.0  # diffusers clamp


def test_rope_table_properties():
    cfg = dit_oracle.DiTConfig.tiny()
    f2 = dit_oracle.rope_table(cfg, 2, 8, 12)
    f8 = dit_oracle.rope_table(cfg, 8, 8, 12)
    assert f2.shape == (1, 1, 2 * 4 * 6, 64) and f2.dtype == torch.complex128
    per = 4 * 6
    # 2 latent frames use temporal positions {0, skip_len - 1} (transformer_chronoedit.py:206-207)
    torch.testing.assert_close(f2[0, 0, :per], f8[0, 0, :per])
    torch.testing.assert_close(f2[0, 0, per:], f8[0, 0, 7 * per:])
    torch.testing.assert_close(f2.abs(), torch.ones_like(f2.abs()))
    with pytest.raises(AssertionError, match="num_frames must be 2 or 8"):
        dit_oracle.rope_table(cfg, 5, 8, 12)


def test_flop_model_matches_survey():
    cfg = dit_oracle.DiTConfig.chronoedit_14b()
    f = dit_oracle.flops_per_forward(cfg, 2, 90, 160)
    assert abs(f / 1e12 - 222.43) < 0.5          # SURVEY.md section 8d
    f8 = dit_oracle.flops_per_forward(cfg, 8, 90, 160)
    assert abs(f8 / 1e12 - 1389.5) < 3.0
    v = vae_oracle.VAEConfig.wan21()
    assert abs(vae_oracle.conv_flops(v, 5, 720, 1280, True) / 1e12 - 41.04) < 0.8
    assert abs(vae_oracle.conv_flops(v, 5, 720, 1280, False) / 1e12 - 24.58) < 0.8
    n = sum(int(torch.tensor(s).prod()) for s in dit_oracle.param_shapes(cfg).values())
    assert abs(n / 1e9 - 16.395) < 0.01


def test_oracle_matches_live_reference(golden_dir):
    """The fp32 output of the reference's ChronoEditTransformer3DModel on these weights and inputs, as stored by make_golden.py."""
    case = cases.DIT_CASES["tiny_t2"]
    y = load_file(os.path.join(golden_dir, "dit_tiny_t2.safetensors"))["out_fp32"]
    sd = cases.dit_weights(case)
    x, t, text, img = cases.dit_inputs(case)
    with torch.no_grad():
        o = dit_oracle.dit_forward(sd, case.cfg, x, t, text, img)
    torch.testing.assert_close(o, y, rtol=0, atol=1e-6)


def test_bench_flop_counters_match_oracle():
    """bench.py restates the algorithmic FLOP counts (so its measured arm never imports oracle/); they must equal the oracle's."""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("_bench_for_test", os.path.join(root, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    for layers, frames, batch in [(40, 2, 2), (1, 8, 1), (0, 2, 1)]:
        assert b.dit_flops_per_forward(layers, frames, 90, 160, 512, 257, batch) == dit_oracle.flops_per_forward(
            dit_oracle.DiTConfig(num_layers=layers), frames, 90, 160, 512, 257, batch=batch)
    cfg = vae_oracle.VAEConfig.wan21()
    assert b.VAE_ENCODE_FLOP == vae_oracle.conv_flops(cfg, 5, 720, 1280, False)
    assert b.VAE_DECODE_FLOP == vae_oracle.conv_flops(cfg, 5, 720, 1280, True)
