#!/usr/bin/env python
"""LoRA golden data, recorded by running the UNMODIFIED reference (its location is taken from $CHRONOEDIT_REFERENCE, see
oracle/ref_loader.py).

    python tests/golden/make_golden_lora.py      # writes tests/golden/LORA_MANIFEST.json

  * converter_wan_key_of_diffusers_key: what the reference's DiffSynth state-dict converter
    (chronoedit_diffsynth/wan_video_dit_chronoedit.py:434-541, `WanModelStateDictConverter.from_diffusers`) renames every
    parameter of the 2-layer oracle DiT to -- the Wan <-> diffusers module map the original-Wan LoRA key style relies on.
  * cli_lora_video: shape and SHA-256 of the bf16 video the UNMODIFIED `ChronoEditPipeline.__call__` makes from the transformer
    mirror after `pipe.load_lora_weights(...)` / `pipe.fuse_lora(lora_scale=0.8)` (tests/test_pipeline_cpu.py); generation
    aborts unless it equals the oracle modules run on the merged weights bit for bit.
"""
from __future__ import annotations

import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import dit_oracle, pipeline_cases as PC, pipeline_oracle as P, ref_loader  # noqa: E402
from tests.test_pipeline_cpu import _cli_lora, _mirror_scheduler, _mirror_transformer, _mirror_vae, _video_sha256  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def converter_key_map():
    names = sorted(dit_oracle.param_shapes(dit_oracle.DiTConfig.tiny()))
    ds = ref_loader.load_reference_diffsynth_dit()
    converted, _ = ds.WanModelStateDictConverter().from_diffusers({k: torch.tensor(float(i)) for i, k in enumerate(names)})
    return {names[int(v)]: wan for wan, v in sorted(converted.items())}


def cli_lora_video():
    case = PC.PIPELINE_CASES["edit_nocfg"]
    dsd, vsd = PC.weights()
    tr = _mirror_transformer(dsd)
    pl = ref_loader.load_reference_pipeline()
    pipe = pl.ChronoEditPipeline(tokenizer=None, text_encoder=None, image_encoder=None, image_processor=None, transformer=tr,
                                 vae=_mirror_vae(vsd), scheduler=_mirror_scheduler(case.sched_shift), disable_guardrails=True)
    pipe.load_lora_weights(_cli_lora(dsd))
    pipe.fuse_lora(lora_scale=0.8)
    merged = {k: v.clone() for k, v in tr.state_dict().items()}
    got = PC.run_reference_pipeline(case, torch.bfloat16, transformer=tr, vae=pipe.vae, scheduler=pipe.scheduler)
    want = PC.run_oracle_pipeline(case, torch.bfloat16, transformer=P.OracleTransformer(merged, PC.DIT_CFG, torch.bfloat16))
    assert torch.equal(got, want), float((got.float() - want.float()).abs().max())
    return {"case": case.name, "lora_scale": 0.8, "dtype": "bfloat16", "shape": list(got.shape), "sha256": _video_sha256(got)}


def main():
    assert ref_loader.reference_available(), "set CHRONOEDIT_REFERENCE to a checkout of the reference"
    torch.set_num_threads(PC.GOLDEN_THREADS)
    manifest = {"torch": torch.__version__, "generated_by": "tests/golden/make_golden_lora.py",
                "converter_wan_key_of_diffusers_key": converter_key_map(), "cli_lora_video": cli_lora_video()}
    with open(os.path.join(OUT, "LORA_MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", os.path.join(OUT, "LORA_MANIFEST.json"))


if __name__ == "__main__":
    main()
