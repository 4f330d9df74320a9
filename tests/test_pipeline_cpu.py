"""Pipeline-level boundary tests that run WITHOUT a GPU (-m "not gpu").

(1) Pin of oracle/pipeline_oracle.py: the UNMODIFIED reference pipeline (chronoedit_diffusers/pipeline_chronoedit.py,
    `ChronoEditPipeline.__call__` :484-812), executed through oracle/diffusers_shim with the reference's own transformer / VAE
    twin / flow-UniPC scheduler, produced the videos stored in tests/golden/pipeline_*.safetensors
    (tests/golden/make_golden_pipeline.py); the restatement driven by the oracle modules must reproduce them bit for bit --
    with and without the temporal-reasoning cut (:700-709) and the two-decode tail (:776-779).
(2) Drop-in surface: the pipeline loop pinned in (1) is run with the three chronoedit_b200 mirrors in place of the oracle's
    objects.  There is no GPU here and the mirrors have no CPU path, so their three native seams (`_native_forward`,
    `_native_encode/_native_decode`, `_native_step`) are stood in for by the oracle -- everything else (constructor surface,
    `.config`, `.dtype`, `temperal_downsample`, argument handling, return types, the scheduler state the pipeline slices in
    place, LoRA loading through `pipe.load_lora_weights / fuse_lora`) is the product code, and the video must equal the
    reference's.  The GPU twin of this test (tests/test_gpu_pipeline.py) runs the real kernels under the same loop.
"""
import hashlib
import json
import os

import pytest
import torch
from safetensors.torch import load_file

from oracle import cases, dit_oracle as D, pipeline_cases as PC, pipeline_oracle as P, unipc_oracle as U, vae_oracle as V

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(autouse=True)
def _golden_thread_count():
    n = torch.get_num_threads()
    torch.set_num_threads(PC.GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", list(PC.PIPELINE_CASES))
def test_pipeline_restatement_is_bit_identical_to_the_unmodified_pipeline(name):
    case = PC.PIPELINE_CASES[name]
    ref = load_file(os.path.join(GOLDEN, f"pipeline_{name}.safetensors"))["video_ref_bf16"]
    ora = PC.run_oracle_pipeline(case, torch.bfloat16)
    assert ref.shape == ora.shape and ref.dtype == ora.dtype
    assert torch.equal(ref, ora), float((ref.float() - ora.float()).abs().max())


@pytest.mark.parametrize("name", list(PC.PIPELINE_CASES))
def test_pipeline_restatement_matches_stored_reference_output(name):
    case = PC.PIPELINE_CASES[name]
    gold = load_file(os.path.join(GOLDEN, f"pipeline_{name}.safetensors"))
    ora = PC.run_oracle_pipeline(case, torch.bfloat16).float()
    ref = gold["video_ref_bf16"].float()
    assert ora.shape == ref.shape
    # same torch build / CPU kernels / thread count -> identical; a different CPU (other bf16 GEMM paths) may flip isolated
    # bf16 ulps
    assert (ora - ref).abs().mean() <= 2e-3 and (ora - ref).abs().max() <= 0.1


# ---------------------------------------------------------------------------------------------------------------------
# (2) the pipeline loop with the mirrors
# ---------------------------------------------------------------------------------------------------------------------
def _mirror_transformer(dsd):
    import chronoedit_b200 as ce

    cfg = PC.DIT_CFG
    m = ce.ChronoEditTransformer3DModel(
        patch_size=cfg.patch_size, num_attention_heads=cfg.num_attention_heads, attention_head_dim=cfg.attention_head_dim,
        in_channels=cfg.in_channels, out_channels=cfg.out_channels, text_dim=cfg.text_dim, freq_dim=cfg.freq_dim, ffn_dim=cfg.ffn_dim,
        num_layers=cfg.num_layers, eps=cfg.eps, image_dim=cfg.image_dim, added_kv_proj_dim=cfg.added_kv_proj_dim)
    m.load_state_dict(cases.to_bf16_state(dsd))

    def native_forward(x, t, txt, img, out, b0, caps, txt_in, img_in):   # stands in for ce_dit_forward_ex
        out.copy_(D.dit_forward(dict(m.state_dict()), cfg, x, t, txt, img))

    m._native_forward = native_forward
    return m


def _mirror_vae(vsd):
    from chronoedit_b200.autoencoder import AutoencoderKLWan

    cfg = PC.VAE_CFG
    m = AutoencoderKLWan(base_dim=cfg.dim, z_dim=cfg.z_dim, dim_mult=tuple(cfg.dim_mult), num_res_blocks=cfg.num_res_blocks,
                         temperal_downsample=tuple(cfg.temperal_downsample))
    m.load_state_dict({k: v.to(torch.bfloat16) for k, v in vsd.items()})

    def native_encode(x, out):   # stands in for ce_vae_encode (moments = mean | logvar; the pipeline only reads the mean)
        out.zero_()
        out[:, : cfg.z_dim] = V.vae_encode(dict(m.state_dict()), cfg, x)

    def native_decode(z, out):   # stands in for ce_vae_decode
        out.copy_(V.vae_decode(dict(m.state_dict()), cfg, z, clamp=m.clamp_output))

    m._native_encode, m._native_decode = native_encode, native_decode
    return m


def _mirror_scheduler(shift):
    import chronoedit_b200 as ce

    s = ce.FlowUniPCMultistepScheduler(shift=shift)

    def native_step(a, t):   # stands in for ce_unipc_step: the oracle's formula list with the oracle's own coefficients
        have_last = t["last_sample"] is not None
        c = U.step_coeffs(s.sigmas, s._step_index, s.num_inference_steps, s.lower_order_nums, s.this_order, have_last, t["sample"].dtype)
        v = t["cond"] if t["uncond"] is None else U.cfg_combine(t["cond"], t["uncond"], a.guidance)
        m_t, x, nxt = U.step_formulas(c, v, t["sample"], t["last_sample"], t["m_prev"], t["m_prev2"])
        t["x0"].copy_(m_t)
        t["prev"].copy_(nxt)
        if t["corrected"] is not None:
            t["corrected"].copy_(x)

    s._native_step = native_step
    return s


@pytest.mark.parametrize("name", list(PC.PIPELINE_CASES))
def test_pipeline_drives_the_mirrors(name):
    case = PC.PIPELINE_CASES[name]
    dsd, vsd = PC.weights()
    ref = load_file(os.path.join(GOLDEN, f"pipeline_{name}.safetensors"))["video_ref_bf16"]
    tr, vae, sch = _mirror_transformer(dsd), _mirror_vae(vsd), _mirror_scheduler(case.sched_shift)
    got = PC.run_oracle_pipeline(case, torch.bfloat16, transformer=tr, vae=vae, scheduler=sch)
    assert got.shape == ref.shape
    assert torch.equal(got, ref), float((got.float() - ref.float()).abs().max())


def _cli_lora(dsd):
    """A seeded LoRA file in diffusers / PEFT key style over six of the projections of every block."""
    g = torch.Generator().manual_seed(5)
    lora = {}
    for k, w in dsd.items():
        if k.endswith(".weight") and any(s in k for s in ("attn1.to_q", "attn1.to_out.0", "attn2.to_k", "attn2.add_v_proj", "ffn.net.0.proj", "ffn.net.2")):
            mod = k[: -len(".weight")]
            lora[f"transformer.{mod}.lora_A.weight"] = (torch.randn(4, w.shape[1], generator=g) * 0.2).bfloat16()
            lora[f"transformer.{mod}.lora_B.weight"] = (torch.randn(w.shape[0], 4, generator=g) * 0.2).bfloat16()
    return lora


def _video_sha256(video):
    return hashlib.sha256(video.contiguous().view(torch.int16).numpy().tobytes()).hexdigest()


def test_cli_lora_lines_work_on_the_mirror():
    """run_inference_diffusers.py:369-376: pipe.load_lora_weights(path); pipe.fuse_lora(lora_scale=s) -- through the
    WanLoraLoaderMixin that ChronoEditPipeline takes both from, into the transformer mirror; the video must equal the oracle
    modules run on the merged weights, and the video the unmodified pipeline made from the same mirror (recorded as a digest
    by tests/golden/make_golden_lora.py)."""
    from oracle.diffusers_shim.diffusers.loaders import WanLoraLoaderMixin

    class Pipe(WanLoraLoaderMixin):
        def __init__(self, transformer):
            self.transformer = transformer

    case = PC.PIPELINE_CASES["edit_nocfg"]
    dsd, vsd = PC.weights()
    lora = _cli_lora(dsd)
    tr = _mirror_transformer(dsd)
    pipe = Pipe(tr)
    pipe.load_lora_weights(lora)
    pipe.fuse_lora(lora_scale=0.8)
    merged = {k: v.clone() for k, v in tr.state_dict().items()}
    base = cases.to_bf16_state(dsd)
    changed = [k for k in merged if not torch.equal(merged[k], base[k])]
    assert len(changed) == len(lora) // 2
    got = PC.run_oracle_pipeline(case, torch.bfloat16, transformer=tr, vae=_mirror_vae(vsd), scheduler=_mirror_scheduler(case.sched_shift))
    want = PC.run_oracle_pipeline(case, torch.bfloat16, transformer=P.OracleTransformer(merged, PC.DIT_CFG, torch.bfloat16))
    assert torch.equal(got, want)
    with open(os.path.join(GOLDEN, "LORA_MANIFEST.json")) as f:
        ref = json.load(f)["cli_lora_video"]
    assert list(got.shape) == ref["shape"] and _video_sha256(got) == ref["sha256"]
