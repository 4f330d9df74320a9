#!/usr/bin/env python
"""Pipeline-level golden vectors: the UNMODIFIED `ChronoEditPipeline.__call__`
(/root/reference/chronoedit_diffusers/pipeline_chronoedit.py:484-812, executed through oracle/diffusers_shim) driving the
reference's OWN modules -- ChronoEditTransformer3DModel (transformer_chronoedit.py), the in-tree Wan VAE twin (wan2pt1.py WanVAE_
behind the AutoencoderKLWan surface) and the flow-matching UniPC scheduler (fm_solvers_unipc.py) -- on seeded tiny weights,
with `prompt_embeds` / `negative_prompt_embeds` / `image_embeds` passed in (the encoders are "next" rows) and guardrails off.

    python tests/golden/make_golden_pipeline.py      # writes tests/golden/pipeline_*.safetensors + PIPELINE_MANIFEST.json

It also requires oracle/pipeline_oracle.py (restatement of the same loop over the oracle restatements of the three
modules) to reproduce every output bit for bit, which is what pins the restatement used on the GPU box.
"""
from __future__ import annotations

import json
import os
import sys

import torch
from safetensors.torch import save_file

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import cases, pipeline_cases, pipeline_oracle, ref_loader  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    assert ref_loader.reference_available(), "run this in the build container (needs /root/reference)"
    torch.set_num_threads(pipeline_cases.GOLDEN_THREADS)
    manifest = {"torch": torch.__version__, "generated_by": "tests/golden/make_golden_pipeline.py", "cases": {}}
    for name, case in pipeline_cases.PIPELINE_CASES.items():
        ref16 = pipeline_cases.run_reference_pipeline(case, torch.bfloat16)
        ref32 = pipeline_cases.run_reference_pipeline(case, torch.float32)
        ora16 = pipeline_cases.run_oracle_pipeline(case, torch.bfloat16)
        ora32 = pipeline_cases.run_oracle_pipeline(case, torch.float32)
        assert ref16.shape == ora16.shape == ref32.shape, (ref16.shape, ora16.shape)
        assert torch.equal(ref16, ora16), (name, float((ref16.float() - ora16.float()).abs().max()))
        d32 = float((ref32.float() - ora32.float()).abs().max())
        assert d32 <= 2e-2, (name, d32)   # fp32 modules, bf16 latents between steps: bf16-ulp flips can appear
        save_file({"video_ref_bf16": ref16.contiguous(), "video_ref_fp32modules": ref32.float().contiguous()},
                  os.path.join(OUT, f"pipeline_{name}.safetensors"))
        manifest["cases"][name] = {
            "shape": list(ref16.shape), "oracle_vs_reference_bf16_equal": True, "oracle_vs_reference_fp32modules_maxabs": d32,
            "bf16_vs_fp32modules_meanabs": float((ref16.float() - ref32.float()).abs().mean()),
            "video_meanabs": float(ref32.float().abs().mean()), "inputs_checksum": pipeline_cases.inputs_checksum(case),
        }
        print(name, manifest["cases"][name], flush=True)
    with open(os.path.join(OUT, "PIPELINE_MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
