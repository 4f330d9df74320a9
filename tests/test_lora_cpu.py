"""CPU tests (-m "not gpu") of `ChronoEditTransformer3DModel.fuse_lora`: the merge arithmetic (W += (B @ A) * s * alpha / r in
the weight dtype), the two key conventions (diffusers / PEFT names and the original Wan names the in-tree loader handles,
chronoedit/_src/models/utils.py:66-190), and the Wan <-> diffusers module map against what the reference's own state-dict
converter (chronoedit_diffsynth/wan_video_dit_chronoedit.py:434-541) made of the same names (tests/golden/make_golden_lora.py)."""
import json
import os

import pytest
import torch

from oracle import dit_oracle as O


def _model():
    import chronoedit_b200 as ce
    cfg = O.DiTConfig.tiny()
    m = ce.ChronoEditTransformer3DModel(num_attention_heads=2, in_channels=36, ffn_dim=cfg.ffn_dim, num_layers=2, image_dim=1280,
                                        added_kv_proj_dim=256)
    g = torch.Generator().manual_seed(0)
    for p in m.parameters():
        p.data.copy_(torch.randn(p.shape, generator=g).to(p.dtype) * 0.05)
    return m


DIFFUSERS_MODULES = ["attn1.to_q", "attn1.to_k", "attn1.to_v", "attn1.to_out.0", "attn2.to_q", "attn2.to_k", "attn2.to_v", "attn2.to_out.0",
                     "attn2.add_k_proj", "attn2.add_v_proj", "ffn.net.0.proj", "ffn.net.2"]
WAN_MODULES = ["self_attn.q", "self_attn.k", "self_attn.v", "self_attn.o", "cross_attn.q", "cross_attn.k", "cross_attn.v", "cross_attn.o",
               "cross_attn.k_img", "cross_attn.v_img", "ffn.0", "ffn.2"]


def _lora(m, rank=4, alpha=8.0, seed=1):
    g = torch.Generator().manual_seed(seed)
    params = dict(m.named_parameters())
    dif, wan = {}, {}
    for blk in range(2):
        for d, w in zip(DIFFUSERS_MODULES, WAN_MODULES):
            W = params[f"blocks.{blk}.{d}.weight"]
            A = (torch.randn(rank, W.shape[1], generator=g) * 0.1).bfloat16()
            B = (torch.randn(W.shape[0], rank, generator=g) * 0.1).bfloat16()
            dif[f"transformer.blocks.{blk}.{d}.lora_A.weight"] = A
            dif[f"transformer.blocks.{blk}.{d}.lora_B.weight"] = B
            dif[f"transformer.blocks.{blk}.{d}.alpha"] = torch.tensor(alpha)
            wan[f"diffusion_model.blocks.{blk}.{w}.lora_down.weight"] = A
            wan[f"diffusion_model.blocks.{blk}.{w}.lora_up.weight"] = B
            wan[f"diffusion_model.blocks.{blk}.{w}.alpha"] = torch.tensor(alpha)
    return dif, wan


def test_fuse_lora_arithmetic_and_key_styles():
    m1, m2 = _model(), _model()
    before = {k: v.clone() for k, v in m1.state_dict().items()}
    dif, wan = _lora(m1)
    assert m1.fuse_lora(dif, lora_scale=0.75) == 24
    assert m2.fuse_lora(wan, lora_scale=0.75) == 24
    after1, after2 = m1.state_dict(), m2.state_dict()
    touched = 0
    for k, w0 in before.items():
        assert torch.equal(after1[k], after2[k]), k   # both key conventions give the same weights
        mod = k[: -len(".weight")] if k.endswith(".weight") else None
        a_key = f"transformer.{mod}.lora_A.weight" if mod else None
        if a_key in dif:
            A, B = dif[a_key], dif[f"transformer.{mod}.lora_B.weight"]
            want = w0 + (B @ A) * (0.75 * 8.0 / 4)                      # PEFT merge, in bf16
            assert torch.equal(after1[k], want), k
            exact = w0.float() + (B.float() @ A.float()) * (0.75 * 8.0 / 4)
            torch.testing.assert_close(after1[k].float(), exact, rtol=2 ** -7, atol=2e-3)
            touched += 1
        else:
            assert torch.equal(after1[k], w0), f"{k} must not change"
    assert touched == 24


def test_fuse_lora_rejects_what_it_cannot_merge():
    from chronoedit_b200 import CEError
    m = _model()
    dif, _ = _lora(m)
    with pytest.raises(CEError):
        m.fuse_lora({"blocks.0.attn1.to_q.lora_A.weight": dif["transformer.blocks.0.attn1.to_q.lora_A.weight"]})
    with pytest.raises(CEError):
        m.fuse_lora({"blocks.0.norm2.diff": torch.zeros(4)})
    with pytest.raises(CEError):
        m.fuse_lora({"blocks.0.attn1.to_q.lora_A.weight": torch.zeros(4, 7), "blocks.0.attn1.to_q.lora_B.weight": torch.zeros(256, 4)})
    with pytest.raises(CEError):
        m.fuse_lora({"blocks.9.attn1.to_q.lora_A.weight": torch.zeros(4, 256), "blocks.9.attn1.to_q.lora_B.weight": torch.zeros(256, 4)})


def test_fuse_lora_is_all_or_nothing():
    """One bad entry anywhere in the file must leave every weight untouched (validation happens before the first update)."""
    from chronoedit_b200 import CEError
    m = _model()
    before = {k: v.clone() for k, v in m.state_dict().items()}
    dif, _ = _lora(m)
    bad = dict(dif)
    bad["transformer.blocks.1.ffn.net.2.lora_B.weight"] = torch.zeros(7, 4, dtype=torch.bfloat16)   # wrong shape, last module
    with pytest.raises(CEError):
        m.fuse_lora(bad)
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]), f"{k} was modified by a rejected fuse"


def test_fuse_lora_non_block_modules_and_peft_adapter_segment():
    """Original-Wan files carry non-block modules (utils.py:214-290); PEFT files carry `.default.` between lora_A/B and weight."""
    m = _model()
    params = dict(m.named_parameters())
    g = torch.Generator().manual_seed(3)
    wan_to_dif = {"time_embedding.0": "condition_embedder.time_embedder.linear_1", "text_embedding.2": "condition_embedder.text_embedder.linear_2",
                  "time_projection.1": "condition_embedder.time_proj", "head.head": "proj_out",
                  "img_emb.proj.1": "condition_embedder.image_embedder.ff.net.0.proj", "img_emb.proj.3": "condition_embedder.image_embedder.ff.net.2"}
    sd, want = {}, {}
    for wan, dif in wan_to_dif.items():
        W = params[dif + ".weight"]
        A = (torch.randn(2, W.shape[1], generator=g) * 0.1).to(W.dtype)
        B = (torch.randn(W.shape[0], 2, generator=g) * 0.1).to(W.dtype)
        sd[f"diffusion_model.{wan}.lora_down.weight"], sd[f"diffusion_model.{wan}.lora_up.weight"] = A, B
        want[dif] = W.data.clone() + (B @ A) * 0.5
    W = params["blocks.1.attn1.to_q.weight"]
    A, B = (torch.randn(2, 256, generator=g) * 0.1).bfloat16(), (torch.randn(256, 2, generator=g) * 0.1).bfloat16()
    sd["transformer.blocks.1.attn1.to_q.lora_A.default.weight"], sd["transformer.blocks.1.attn1.to_q.lora_B.default.weight"] = A, B
    want["blocks.1.attn1.to_q"] = W.data.clone() + (B @ A) * 0.5
    assert m.fuse_lora(sd, lora_scale=0.5) == len(want)
    for mod, w in want.items():
        assert torch.equal(dict(m.named_parameters())[mod + ".weight"].data, w), mod


def test_diffusers_style_load_then_fuse():
    """`pipe.load_lora_weights(x); pipe.fuse_lora(lora_scale=s)` reaches the transformer as load_lora_adapter(state_dict,
    prefix="transformer", ...) + fuse_lora(s, safe_fusing=..., adapter_names=...) ([diffusers-mem]; run_inference_diffusers.py:369-376)."""
    from chronoedit_b200 import CEError
    m1, m2 = _model(), _model()
    dif, _ = _lora(m1)
    m1.fuse_lora(dif, lora_scale=0.75)
    m2.load_lora_adapter(dif, prefix="transformer", adapter_name="lora")
    assert m2.fuse_lora(0.75, safe_fusing=True, adapter_names=None) == 24
    for (k, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    with pytest.raises(CEError):
        m2.fuse_lora(0.75)   # already merged: nothing left to fuse, and certainly not twice


def test_wan_to_diffusers_module_map_matches_reference_converter(golden_dir):
    import chronoedit_b200 as ce
    with open(os.path.join(golden_dir, "LORA_MANIFEST.json")) as f:
        to_wan = json.load(f)["converter_wan_key_of_diffusers_key"]
    for wan, dif in ce.ChronoEditTransformer3DModel._WAN_TO_DIFFUSERS:
        assert to_wan[f"blocks.0.{dif}.weight"] == f"blocks.0.{wan}.weight", (wan, dif)
    for wan, dif in ce.ChronoEditTransformer3DModel._WAN_TO_DIFFUSERS_GLOBAL.items():
        assert to_wan[f"{dif}.weight"] == f"{wan}.weight", (wan, dif)


def test_new_weights_drop_the_context_cache():
    """The step-invariant context cache is keyed on the conditioning tensors only, so anything that changes the weights has to empty
    it: load_state_dict (also mid-session), fuse_lora (tested above through its effect on the weights), .to()."""
    import chronoedit_b200 as ce

    m = ce.ChronoEditTransformer3DModel(num_attention_heads=2, in_channels=36, ffn_dim=256, num_layers=1, image_dim=1280, added_kv_proj_dim=256,
                                        text_dim=64, cache_context=True)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    m._ctx_cache = [dict(txt=None, img=None, txt_v=None, img_v=None, buf=None)]
    m._graphs = {"k": object()}
    m.load_state_dict(sd)
    assert m._ctx_cache == [] and m._graphs == {}
    m._ctx_cache = [dict(txt=None, img=None, txt_v=None, img_v=None, buf=None)]
    m.to(torch.bfloat16)
    assert m._ctx_cache == []
