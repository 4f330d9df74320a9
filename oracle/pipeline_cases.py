"""Seeded pipeline-level parity cases (BASELINE.json configs[0] scale: 2-layer / dim-256 DiT + a narrow Wan VAE) and the
runners that push them through (a) the UNMODIFIED reference pipeline with the reference's own modules (build container only),
(b) the pipeline restatement with the oracle modules (CPU or CUDA), (c) either of those loops with the chronoedit_b200
mirrors.  TEST INFRASTRUCTURE ONLY (oracle/__init__.py)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict

import torch

from . import cases, pipeline_oracle as P
from . import dit_oracle as D
from . import vae_oracle as V


@dataclass
class PipelineCase:
    name: str
    height: int
    width: int
    num_frames: int
    steps: int = 4
    guidance: float = 5.0
    enable_temporal_reasoning: bool = False
    num_temporal_reasoning_steps: int = 0
    sched_shift: float = 3.0
    text_valid: int = 37
    seed: int = 2024


PIPELINE_CASES: Dict[str, PipelineCase] = {
    c.name: c
    for c in [
        # one edit: 5 pixel frames -> 2 latent frames, 4 steps, CFG 5.0 (configs[0] plumbing case, small picture)
        PipelineCase("edit_5f", height=128, width=192, num_frames=5),
        # temporal reasoning with the in-loop cut at step 2 (pipeline_chronoedit.py:700-709) and the two-decode tail (:776-779)
        PipelineCase("reason_cut", height=64, width=96, num_frames=29, enable_temporal_reasoning=True, num_temporal_reasoning_steps=2),
        # the CLI default: reasoning steps == inference steps, the cut never fires, two decodes of 2 and 7 latent frames
        PipelineCase("reason_full", height=64, width=96, num_frames=29, enable_temporal_reasoning=True, num_temporal_reasoning_steps=4),
        # distilled-LoRA style run: guidance 1.0 -> one forward per step (run_inference_diffusers.py:179-189)
        PipelineCase("edit_nocfg", height=64, width=96, num_frames=5, steps=3, guidance=1.0, sched_shift=2.0),
    ]
}

DIT_CFG = D.DiTConfig.tiny()
VAE_CFG = V.VAEConfig.tiny(32)
# torch's bf16 matrix products on the CPU (oneDNN) round differently with the number of intra-op threads, and the difference
# grows over the denoising steps; the stored pipeline videos are made and compared with this many threads
GOLDEN_THREADS = 8


def weights():
    return D.random_state_dict(DIT_CFG, seed=21), V.random_state_dict(VAE_CFG, seed=22)


def inputs(case: PipelineCase):
    g = torch.Generator(device="cpu").manual_seed(case.seed)
    image = torch.rand(1, 3, case.height, case.width, generator=g) * 2 - 1          # preprocessed image in [-1, 1]
    prompt = torch.randn(1, 512, DIT_CFG.text_dim, generator=g)
    prompt[:, case.text_valid:] = 0
    negative = torch.randn(1, 512, DIT_CFG.text_dim, generator=g)
    negative[:, 11:] = 0
    image_embeds = torch.randn(1, 257, DIT_CFG.image_dim, generator=g)
    tl = (case.num_frames - 1) // 4 + 1
    latents = torch.randn(1, 16, tl, case.height // 8, case.width // 8, generator=g)
    return image, prompt, negative, image_embeds, latents


def inputs_checksum(case: PipelineCase) -> float:
    return cases.checksum(torch.cat([t.flatten()[:65536] for t in inputs(case)]))


def _cast_dit(sd, dtype):
    return sd if dtype == torch.float32 else cases.to_bf16_state(sd)


def _call_kwargs(case: PipelineCase):
    return dict(height=case.height, width=case.width, num_frames=case.num_frames, num_inference_steps=case.steps,
                guidance_scale=case.guidance, enable_temporal_reasoning=case.enable_temporal_reasoning,
                num_temporal_reasoning_steps=case.num_temporal_reasoning_steps)


def run_reference_pipeline(case: PipelineCase, dtype: torch.dtype, transformer=None, vae=None, scheduler=None) -> torch.Tensor:
    """The UNMODIFIED ChronoEditPipeline.__call__ (needs /root/reference).  By default with the reference's own modules; any of
    the three can be replaced (e.g. by a chronoedit_b200 mirror) to exercise the drop-in boundary."""
    from tests.golden.make_golden import build_reference_dit

    from . import ref_loader

    pl = ref_loader.load_reference_pipeline()
    dsd, vsd = weights()
    if transformer is None:
        transformer = build_reference_dit(ref_loader.load_reference_dit(), DIT_CFG)
        transformer.load_state_dict(dsd)
        if dtype != torch.float32:
            transformer.to(dtype)
            transformer.load_state_dict(_cast_dit(dsd, dtype), assign=True)
    if vae is None:
        ref_vae = ref_loader.load_reference_vae()
        m = ref_vae.WanVAE_(dim=VAE_CFG.dim, z_dim=VAE_CFG.z_dim, dim_mult=list(VAE_CFG.dim_mult), num_res_blocks=VAE_CFG.num_res_blocks,
                            attn_scales=[], temperal_downsample=list(VAE_CFG.temperal_downsample), dropout=0.0).eval()
        m.load_state_dict(vsd)
        vae = P.RefVAEAdapter(m.to(dtype))
    if scheduler is None:
        scheduler = ref_loader.load_reference_unipc().FlowUniPCMultistepScheduler(shift=case.sched_shift)
    pipe = pl.ChronoEditPipeline(tokenizer=None, text_encoder=None, image_encoder=None, image_processor=None, transformer=transformer,
                                 vae=vae, scheduler=scheduler, disable_guardrails=True)
    image, prompt, negative, image_embeds, latents = inputs(case)
    # `image` must be given (it is preprocessed unconditionally, :673) and cannot be combined with image_embeds (:350-354), so the
    # CLIP encoder is stood in for by a stub that returns the seeded embeddings as hidden_states[-2] (:246-254)
    pipe.image_processor = lambda images, return_tensors: _Batch()
    pipe.image_encoder = lambda **kw: type("O", (), {"hidden_states": [None, image_embeds, None]})()
    out = pipe(image=image, prompt_embeds=prompt, negative_prompt_embeds=negative if case.guidance > 1 else None, latents=latents,
               output_type="pt", return_dict=False, **_call_kwargs(case))[0]
    return out


class _Batch(dict):
    def to(self, device):
        return self


def run_oracle_pipeline(case: PipelineCase, dtype: torch.dtype, device="cpu", transformer=None, vae=None, scheduler=None) -> torch.Tensor:
    """oracle/pipeline_oracle.run_pipeline with the oracle modules (default) or any replacements; returns what the reference call
    returns for output_type="pt": [B, T, 3, H, W] in [0, 1]."""
    dsd, vsd = weights()
    dev = torch.device(device)
    if transformer is None:
        transformer = P.OracleTransformer({k: v.to(dev) for k, v in _cast_dit(dsd, dtype).items()}, DIT_CFG, dtype)
    if vae is None:
        vae = P.OracleVAE({k: v.to(dev, dtype) for k, v in vsd.items()}, VAE_CFG, dtype)
    if scheduler is None:
        scheduler = P.OracleScheduler(shift=case.sched_shift)
    image, prompt, negative, image_embeds, latents = (t.to(dev) for t in inputs(case))
    video = P.run_pipeline(transformer, vae, scheduler, image, prompt, negative if case.guidance > 1 else None, image_embeds,
                           latents=latents, device=dev, **_call_kwargs(case))
    return postprocess_pt(video)


def postprocess_pt(video: torch.Tensor) -> torch.Tensor:
    """VideoProcessor.postprocess_video(video, "pt"): per sample [C,T,H,W] -> [T,C,H,W], (x/2 + 0.5).clamp(0,1), stacked."""
    return torch.stack([(v.permute(1, 0, 2, 3) * 0.5 + 0.5).clamp(0, 1) for v in video])
