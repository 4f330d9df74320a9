"""CPU tests (-m "not gpu") of the sampling-glue row: the oracle restatement of FlowUniPCMultistepScheduler reproduces the
golden vectors recorded from the unmodified reference (tests/golden/make_golden_unipc.py); the product mirror's host-side
logic (sigma schedule, per-step scalars, bookkeeping, error behaviour) agrees with both."""
import json
import os

import numpy as np
import pytest
import torch
from safetensors.torch import load_file

from oracle import unipc_oracle
from oracle.unipc_cases import UNIPC_CASES, case_inputs


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def _run_oracle(case, cuda_semantics=False):
    o = unipc_oracle.UniPCOracle(shift=1.0, cuda_semantics=cuda_semantics)
    o.set_timesteps(case.steps, shift=case.shift)
    x, cond, uncond = case_inputs(case)
    outs = []
    for i in range(case.steps):
        if case.cut_at is not None and i == case.cut_at:
            x = x[:, :, [0, -1]]
            o.cut_frames()
        c, u = cond[i], uncond[i]
        if case.cut_at is not None and i >= case.cut_at:
            c, u = c[:, :, [0, -1]], u[:, :, [0, -1]]
        v = unipc_oracle.cfg_combine(c, u, case.guidance, cuda_semantics) if case.guidance is not None else c
        x = o.step(v, x)
        outs.append(x)
    return o, outs


@pytest.mark.parametrize("name", sorted(UNIPC_CASES))
def test_oracle_matches_golden_bit_exact(name, golden_dir):
    case = UNIPC_CASES[name]
    gold = load_file(os.path.join(golden_dir, f"unipc_{name}.safetensors"))
    o, outs = _run_oracle(case)
    assert torch.equal(o.sigmas, gold["sigmas"]) and torch.equal(o.timesteps, gold["timesteps"])
    for i, x in enumerate(outs):
        g = gold[f"step{i:02d}"]
        assert x.dtype == g.dtype and x.shape == g.shape
        assert torch.equal(_bits(x), _bits(g)), f"{name}: step {i} differs from the reference"


def test_oracle_matches_live_reference(golden_dir):
    """The reference scheduler stepped by the pipeline's own guidance combine (pipeline_chronoedit.py:736), as stored by
    make_golden_unipc.py."""
    case = UNIPC_CASES["bf16_cfg_10step"]
    gold = load_file(os.path.join(golden_dir, "unipc_bf16_cfg_10step.safetensors"))
    _, outs = _run_oracle(case)
    for i in range(case.steps):
        assert torch.equal(_bits(gold[f"step{i:02d}"]), _bits(outs[i]))


def test_cuda_scalar_semantics_distance_is_as_recorded(golden_dir):
    """torch's CUDA kernels keep fp32 coefficients at full precision and multiply by 1/r_k where its CPU kernels round the
    coefficient to the tensor dtype first and divide (oracle/unipc_oracle.py header).  With bf16 latents that is a visible
    difference between a CPU and a GPU run OF THE REFERENCE ITSELF (coefficients lose 8 of their 24 bits on CPU and the update
    subtracts nearly equal terms).  The golden vectors are a CPU run; the manifest records how far the emulated CUDA semantics
    land from them, and the GPU tests bound the kernel-vs-golden distance by that number.  With fp32 latents and fp32 model
    outputs only the division differs and the distance is one rounding."""
    man = json.load(open(os.path.join(golden_dir, "UNIPC_MANIFEST.json")))["cases"]
    for name, case in UNIPC_CASES.items():
        _, a = _run_oracle(case, cuda_semantics=False)
        _, b = _run_oracle(case, cuda_semantics=True)
        n_diff = sum(int((x != y).sum()) for x, y in zip(a, b))
        max_diff = max(float((x.float() - y.float()).abs().max()) for x, y in zip(a, b))
        assert n_diff == man[name]["elements_changed_by_cuda_semantics"]
        assert max_diff == man[name]["max_abs_change_by_cuda_semantics"]
        if case.sample_dtype == torch.float32 and case.model_dtype == torch.float32:
            assert max_diff <= 2.5e-7 * max(1.0, max(float(x.abs().max()) for x in a))


# ---------------------------------------------------------------------------------------------- product mirror, host side
def test_mirror_schedule_matches_reference_schedule(golden_dir):
    from chronoedit_b200.scheduler import FlowUniPCMultistepScheduler
    for name, case in UNIPC_CASES.items():
        gold = load_file(os.path.join(golden_dir, f"unipc_{name}.safetensors"))
        s = FlowUniPCMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
        s.set_timesteps(case.steps, device="cpu", shift=case.shift)
        assert torch.equal(s.sigmas, gold["sigmas"]) and torch.equal(s.timesteps, gold["timesteps"])
        assert s.timesteps.dtype == torch.int64 and s.sigmas.device.type == "cpu"
        assert s.model_outputs == [None, None] and s.last_sample is None and s.step_index is None and s.order == 1


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("steps,shift", [(8, 2.0), (50, 5.0), (1, 2.0), (2, 3.0)])
def test_mirror_step_scalars_match_oracle(steps, shift, dtype):
    """Per-step scalars the kernel receives == the oracle's (which reproduces the reference bit for bit)."""
    from chronoedit_b200 import _lib
    from chronoedit_b200.scheduler import FlowUniPCMultistepScheduler
    s = FlowUniPCMultistepScheduler(shift=1)
    s.set_timesteps(steps, device="cpu", shift=shift)
    sig, _ = unipc_oracle.flow_sigmas(steps, shift)
    lower, prev_order = 0, 1
    for i in range(steps):
        have_last = i > 0
        s.last_sample = torch.zeros(1) if have_last else None
        s.this_order, s.lower_order_nums = prev_order, lower
        a = _lib.UniPCStepArgsC()
        order = s._fill_coefficients(a, i, dtype)
        c = unipc_oracle.step_coeffs(sig, i, steps, lower, prev_order, have_last, dtype)
        f32 = lambda v: float(np.float32(v))  # noqa: E731
        assert order == c.p_order and bool(a.use_corrector) == c.use_corrector
        assert (a.sigma, a.p_x, a.p_m0, a.p_bh) == (f32(c.sigma), f32(c.p_x), f32(c.p_m0), f32(c.p_bh))
        assert np.signbit(a.p_zero) == np.signbit(c.p_zero) and a.p_zero == c.p_zero
        if order == 2:
            assert a.p_inv_rk == f32(np.float32(1.0) / np.float32(c.p_rk))
        if c.use_corrector:
            assert a.c_order == c.c_order and (a.c_x, a.c_m0, a.c_bh) == (f32(c.c_x), f32(c.c_m0), f32(c.c_bh))
            if c.c_order == 2:
                assert (a.c_rho0, a.c_rho1) == (f32(c.c_rho0), f32(c.c_rho1))
                assert a.c_inv_rk == f32(np.float32(1.0) / np.float32(c.c_rk))
        prev_order, lower = order, min(lower + 1, 2)


def test_mirror_rejects_what_is_not_built():
    from chronoedit_b200.scheduler import FlowUniPCMultistepScheduler
    for kw in ({"solver_order": 3}, {"thresholding": True}, {"predict_x0": False}, {"solver_type": "bh1"}, {"use_dynamic_shifting": True},
               {"disable_corrector": [0]}, {"final_sigmas_type": "sigma_min"}, {"prediction_type": "epsilon"}):
        with pytest.raises(NotImplementedError):
            FlowUniPCMultistepScheduler(**kw)
    with pytest.raises(NotImplementedError):   # same error the reference raises (fm_solvers_unipc.py:110-116)
        FlowUniPCMultistepScheduler(solver_type="nope")
    assert FlowUniPCMultistepScheduler(solver_type="midpoint").config.solver_type == "bh2"   # :111-113


def test_mirror_has_no_cpu_path():
    from chronoedit_b200 import _lib
    from chronoedit_b200.scheduler import FlowUniPCMultistepScheduler
    s = FlowUniPCMultistepScheduler(shift=1)
    x = torch.zeros(1, 16, 2, 4, 6)
    with pytest.raises(ValueError):   # fm_solvers_unipc.py:692-695
        s.step(x, 999, x)
    s.set_timesteps(4, device="cpu", shift=2.0)
    with pytest.raises(_lib.CEError):
        s.step(x, s.timesteps[0], x)
