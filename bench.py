#!/usr/bin/env python
"""Benchmark of the ChronoEdit denoising hot path (BASELINE.json metric: DiT denoising steps/sec at 14B, 720x1280,
5 pixel frames = 2 latent frames).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one iteration of the sampling loop of ChronoEditPipeline.__call__ (pipeline_chronoedit.py:695-753) for ONE
edit with classifier-free guidance: two DiT forwards (prompt / negative prompt — evaluated as one batch-2 call, which the
batch-invariance test proves equal to two batch-1 calls), the CFG combine and the latent update.  Workload = configs[1]:
ChronoEdit-14B (40 layers, dim 5120, ffn 13824), latent [1,36,2,90,160] -> 7200 tokens, 512 text + 257 image tokens,
random-init bf16 weights, synthetic inputs.  With N GPUs every rank runs its own independent edit (data parallel over a
batch of N edits, weak scaling); rank 0 initialises the weights and they are replicated with ONE NCCL broadcast; there
is no per-step collective.

Printed JSON (one line, rank 0):
  value     steps/s summed over ranks, inputs resident in HBM, timed with CUDA events, max over ranks
  e2e       the same step through the host-buffer C-ABI call (ce_dit_forward_host): pinned-host inputs H2D every step,
            sample D2H every step, CFG combine + latent update on the host
  roofline  the dominant kernel class (tcgen05 GEMM): algorithmic FLOPs / device time of those launches measured live
            with CUDA events inside the timed region, against MEASURED_PEAKS.json bf16_tflops_sustained
  cpu_baseline  the oracle (CPU restatement of the reference) timed on the host cores on a bounded sample
--impl reference times that CPU path alone with the same metric/config (the reference has no faster path on this box).

--dump-outputs DIR writes what the last timed step computed on rank 0 as float32 .npy files: noise_pred.npy (the batch-2 DiT
output, conditional then unconditional) and latents.npy (the latents the guided scheduler step returned).  Weights and inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "dit_denoising_steps_per_sec_14B_720p_5frame"
FRAMES, LAT_H, LAT_W, TEXT_LEN = 2, 90, 160, 512
GUIDANCE = 5.0


def model_config(layers: int):
    return dict(patch_size=(1, 2, 2), num_attention_heads=40, attention_head_dim=128, in_channels=36, out_channels=16,
                text_dim=4096, freq_dim=256, ffn_dim=13824, num_layers=layers, image_dim=1280, added_kv_proj_dim=5120)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------------------
# CPU side: the oracle on a bounded sample (cpu_baseline of our arm, and the whole of --impl reference)
# --------------------------------------------------------------------------------------------------------------
def cpu_reference_step_rate(reps: int, warmup: int = 0):
    """Times ONE ChronoEditTransformerBlock at the FULL BASELINE size -- 14B width (dim 5120, 40 heads, ffn 13824), all 7200 tokens of
    the 720p / 2-latent-frame sequence, 769 context tokens -- in fp32 on the host cores with the oracle, `reps` times (each ~3-10 s).
    A denoising step with CFG is 2 forwards x 40 such blocks (identical work; the embedders / head are < 0.1 %), so the step rate is
    1 / (80 x the measured block time): the only scaling is the count of identical blocks, no token-count or FLOP extrapolation.
    Returns (steps_per_sec, seconds per block list, threads, description)."""
    import torch

    from oracle import dit_oracle as O

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.DiTConfig.chronoedit_14b()
    D = cfg.inner_dim
    one = O.DiTConfig(num_layers=1)
    g = torch.Generator().manual_seed(0)
    sd = {k: v for k, v in O.random_state_dict(one, seed=0).items() if k.startswith("blocks.0.")}
    Ls = 7200
    x = torch.randn(1, Ls, D, generator=g)
    ctx = torch.randn(1, 257 + 512, D, generator=g)
    temb6 = torch.randn(1, 6, D, generator=g) * 0.1
    freqs = O.rope_table(cfg, 2, 90, 160)
    times = []
    with torch.no_grad():
        # give the reference its best thread count (oversubscribed SMT threads often hurt torch's CPU GEMMs)
        best = None
        x_probe, f_probe = x[:, :1800], freqs[:, :, :1800]
        for n in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
            torch.set_num_threads(n)
            t0 = time.perf_counter()
            O.block(sd, 0, one, x_probe, ctx, temb6, f_probe)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, n)
        cores = best[1]
        torch.set_num_threads(cores)
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            O.block(sd, 0, one, x, ctx, temb6, freqs)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    t_block = statistics.mean(times)
    step_s = 2 * 40 * t_block
    desc = (f"one full 14B-width DiT block (oracle, fp32) on all 7200 tokens, measured {reps}x ({t_block:.2f} s each), {cores} threads; "
            f"step = 2 CFG forwards x 40 identical blocks = 80 x the measured block")
    return 1.0 / step_s, times, cores, desc


def cpu_extras(threads: int):
    """Two more measured CPU datapoints for the cpu_baseline object (BASELINE.md section 4): the first chunk of a 720p VAE decode
    (latent frame 0 -> pixel frame 0, Wan2.1 width, oracle, fp32) and BASELINE configs[0] end to end (2-layer / dim-256 DiT,
    4 steps with CFG on a [1,36,2,64,64] latent + VAE bookends at 64x64 px through the pipeline restatement)."""
    import torch

    from oracle import pipeline_cases as PC
    from oracle import vae_oracle as V

    torch.set_num_threads(threads)
    out = {}
    cfg = V.VAEConfig.wan21()
    sd = V.random_state_dict(cfg, seed=1)
    z = torch.randn(1, 16, 1, 90, 160, generator=torch.Generator().manual_seed(2))
    t0 = time.perf_counter()
    V.vae_decode(sd, cfg, z)
    out["vae_decode_720p_first_frame_s"] = round(time.perf_counter() - t0, 2)
    case = PC.PIPELINE_CASES["edit_5f"]
    t0 = time.perf_counter()
    PC.run_oracle_pipeline(case, torch.float32)
    dt = time.perf_counter() - t0
    out["config0_edit_s"] = round(dt, 2)
    out["config0_steps_per_s"] = round(case.steps / dt, 3)
    out["config0_note"] = "2-layer/dim-256 DiT, 4 CFG steps + VAE encode/decode, 128x192 px, fp32, oracle pipeline restatement (whole edit, measured)"
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    rate, times, cores, desc = cpu_reference_step_rate(args.steps, args.warmup)
    ms_per_step = 1000.0 / rate
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": ("configs[1]: ChronoEdit-14B single edit, 720x1280, 5 px frames -> latent [1,36,2,90,160] (7200 tokens), "
                                "512 text + 257 image tokens, CFG 5.0 (2 forwards/step)"),
                   "sample_per_step": "one full 14B-width block on all 7200 tokens (measured); step = 80 identical blocks", "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": rate, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(time.perf_counter() - t0, 2),
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------------------
# Algorithmic work (SURVEY.md section 8d), restated here so that the measured arm does not touch oracle/ at all:
# 2*MAC for every Linear, 4*Lq*Lk*D for every attention; tests/test_oracle.py checks these against the oracle's own counters.
def dit_flops_per_forward(layers: int, frames: int, lat_h: int, lat_w: int, text_len: int, image_len: int, batch: int) -> float:
    D, Fd, cin, cout, text_dim, image_dim, freq_dim = 5120, 13824, 36, 16, 4096, 1280, 256
    L = frames * (lat_h // 2) * (lat_w // 2)
    per_block = (2 * L * D * 3 * D + 4 * L * L * D + 2 * L * D * D            # self: q,k,v / SDPA / out
                 + 2 * L * D * D + 2 * text_len * D * 2 * D + 2 * image_len * D * 2 * D   # cross: q / text k,v / image k,v
                 + 4 * L * (text_len + image_len) * D + 2 * L * D * D          # cross: SDPA / out
                 + 2 * 2 * L * D * Fd)                                          # ffn
    embed = (2 * L * cin * 4 * D + 2 * L * D * cout * 4 + 2 * text_len * (text_dim * D + D * D)
             + 2 * image_len * (image_dim ** 2 + image_dim * D) + 2 * (freq_dim * D + D * D + D * 6 * D))
    return float(batch) * (layers * per_block + embed)


VAE_ENCODE_FLOP = 24577494220800.0   # conv FLOPs of one 5 x 720 x 1280 encode / decode (SURVEY 8d: 24.58 / 41.04 TFLOP)
VAE_DECODE_FLOP = 41036724633600.0


def traffic(kernel: str, field: str = "dram_bytes"):
    """Per-launch DRAM traffic of a kernel class from profiles/traffic.json (written by scripts/summarize_profiles.py from the
    committed `ncu --set full` captures); None when there is no capture for it."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        d = json.load(f)
    return (d.get(kernel) or {}).get(field)


def library_bar_step_rate(model, d_in, d_text, d_img, dev, layers: int, steps: int = 2):
    import torch
    from torch.nn.attention import SDPBackend, sdpa_kernel

    from oracle import dit_oracle as O

    cfg = O.DiTConfig(num_layers=layers)
    sd = dict(model.state_dict())   # the mirror's own parameters (views of the fused buffers): no second copy of the weights
    x = d_in.expand(2, -1, -1, -1, -1).contiguous()
    t = torch.tensor([500, 500], device=dev)
    lat = d_in[:, :16].clone()
    out = {}
    for name, backends in (("sdpa_cudnn", [SDPBackend.CUDNN_ATTENTION, SDPBackend.MATH]), ("sdpa_default", None)):
        def step():
            with torch.no_grad():
                o = O.dit_forward(sd, cfg, x, t, d_text, d_img)
                v = o[1:2] + GUIDANCE * (o[0:1] - o[1:2])
                return (lat - 0.02 * v).to(torch.bfloat16)
        try:
            ctx = sdpa_kernel(backends) if backends else None
            if ctx:
                ctx.__enter__()
            step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            if ctx:
                ctx.__exit__(None, None, None)
            out[name] = {"ms_per_step": e0.elapsed_time(e1) / steps, "steps_per_s": steps / (e0.elapsed_time(e1) / 1000.0)}
        except Exception as e:  # noqa: BLE001
            out[name] = {"error": str(e)[:160]}
    best = max((v["steps_per_s"] for v in out.values() if "steps_per_s" in v), default=None)
    return {"value": best, "unit": "steps/s", "what": "oracle restatement of the reference on this GPU, torch eager bf16 (cuBLAS + SDPA + ATen), same weights / step",
            "backends": out, "steps": steps}


def init_weights_(model, seed: int):
    """Random-init weights of the 14B architecture directly on the device (there is no checkpoint on the box):
    Linear ~ N(0, 0.02), norms ~ 1 + 0.1 N, scale_shift_table ~ N(0,1)/sqrt(D) (as transformer_chronoedit.py:265, 393)."""
    import math

    import torch

    g = torch.Generator(device=model.device).manual_seed(seed)
    D = model.config.num_attention_heads * model.config.attention_head_dim
    for n, p in model.named_parameters():
        if n.endswith("scale_shift_table"):
            p.data.normal_(0, 1.0 / math.sqrt(D), generator=g)
        elif ".norm" in n and n.endswith("weight"):
            p.data.normal_(0, 0.1, generator=g).add_(1.0)
        elif ".norm" in n and n.endswith("bias"):
            p.data.normal_(0, 0.1, generator=g)
        else:
            p.data.normal_(0, 0.02, generator=g)


def run_ours(args):
    import torch
    import torch.distributed as dist

    import chronoedit_b200 as ce
    from chronoedit_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus or world == 1, f"WORLD_SIZE {world} != --gpus {args.gpus}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = model_config(args.layers)
    model = ce.ChronoEditTransformer3DModel(**cfg, device=dev, cache_context=not args.no_context_cache)
    # weights: rank 0 initialises, ONE broadcast replicates them (the only collective on the path)
    t_b0 = time.perf_counter()
    if rank == 0:
        init_weights_(model, seed=0)
    model.pack_weights()
    bcast_bytes = 0
    if world > 1:
        from chronoedit_b200 import parallel

        bcast_bytes = parallel.broadcast_module_weights(model, src=0)
        torch.cuda.synchronize()
    t_bcast = time.perf_counter() - t_b0

    # synthetic per-edit inputs (different on every rank: independent edits)
    g = torch.Generator(device="cpu").manual_seed(42 + rank)
    B = 2  # CFG pair
    latents = torch.randn(1, 16, FRAMES, LAT_H, LAT_W, generator=g)
    cond = torch.randn(1, 20, FRAMES, LAT_H, LAT_W, generator=g)
    cond[:, :4] = 0
    cond[:, :4, 0] = 1  # mask channels: frame 0 = 1 (pipeline_chronoedit.py:447-453)
    text = torch.randn(2, TEXT_LEN, 4096, generator=g)
    text[0, 120:] = 0
    text[1, 40:] = 0
    img = torch.randn(1, 257, 1280, generator=g).expand(2, -1, -1).contiguous()
    sigmas = torch.linspace(1.0, 0.0, 51)
    sigmas = 5.0 * sigmas / (1 + 4.0 * sigmas)  # flow shift 5 (run_inference_diffusers.py:203-207)

    d_lat = latents.to(dev)
    d_cond = cond.to(dev, torch.bfloat16)
    d_text = text.to(dev, torch.bfloat16)
    d_img = img.to(dev, torch.bfloat16)

    # The loop body of ChronoEditPipeline.__call__ (pipeline_chronoedit.py:693-739) on device-resident tensors: model input =
    # cat([latents, condition]) in bf16, ONE batch-2 DiT call for the CFG pair, then ONE fused launch for the guidance combine
    # + UniPC flow-matching scheduler step + the latent channels of the next model input (chronoedit_b200/scheduler.py).
    from chronoedit_b200.scheduler import FlowUniPCMultistepScheduler

    sched = FlowUniPCMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
    d_lat = d_lat.to(torch.bfloat16)   # the diffusers pipeline keeps bf16 latents (pipeline_chronoedit.py:676-687)
    d_in = torch.cat([d_lat, d_cond], dim=1).contiguous()

    last = {}

    def device_step(i):
        nonlocal d_lat
        if sched.step_index is None or sched.step_index >= 50:
            sched.set_timesteps(50, device=dev, shift=5.0)   # flow shift 5 (run_inference_diffusers.py:203-207)
        t = sched.timesteps[sched.step_index or 0]
        out = model(d_in.expand(2, -1, -1, -1, -1), t.expand(2), d_text, d_img, return_dict=False)[0]
        d_lat = sched.step_cfg(out[0:1], out[1:2], GUIDANCE, t, d_lat, model_input_out=d_in)
        if args.dump_outputs:
            last["noise_pred"], last["latents"] = out, d_lat

    # host-buffer (e2e) step = the SAME loop body through the host-facing call: every step the model input (built on the host from
    # the host copy of the latents), the timestep and the prompt / image embeddings go pinned-host -> device inside
    # ce_dit_forward_host_ex, the DiT runs, the sample comes back device -> host, the fused CFG + UniPC step (ce_unipc_step)
    # consumes the sample on the device, and the new latents are read back to the host (they are next step's input).
    h_x = torch.empty(2, 36, FRAMES, LAT_H, LAT_W, dtype=torch.bfloat16).pin_memory()
    h_text = text.to(torch.bfloat16).pin_memory()
    h_img = img.to(torch.bfloat16).pin_memory()
    h_out = torch.empty(2, 16, FRAMES, LAT_H, LAT_W, dtype=torch.bfloat16).pin_memory()
    h_lat = latents.to(torch.bfloat16).pin_memory()
    h_cond = cond.to(torch.bfloat16)
    h_x[:, 16:] = h_cond
    h2d = h_x.numel() * 2 + h_text.numel() * 2 + h_img.numel() * 2 + B * 4
    d2h = h_out.numel() * 2 + h_lat.numel() * 2
    sched_h = FlowUniPCMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
    e2e_state = {"lat": latents.to(dev, torch.bfloat16)}

    def host_step(i):
        if sched_h.step_index is None or sched_h.step_index >= 50:
            sched_h.set_timesteps(50, device="cpu", shift=5.0)
            e2e_state["lat"] = h_lat.to(dev, non_blocking=True)
        t = sched_h.timesteps[sched_h.step_index or 0]
        h_x[0, :16].copy_(h_lat[0])
        h_x[1, :16].copy_(h_lat[0])
        _, d_sample = model.forward_host(h_x, t.expand(2), h_text, h_img, out=h_out, return_device_sample=True)
        e2e_state["lat"] = sched_h.step_cfg(d_sample[0:1], d_sample[1:2], GUIDANCE, t, e2e_state["lat"])
        h_lat.copy_(e2e_state["lat"], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sampler=None, profile=False):
        for i in range(warmup):
            fn(i)
        barrier()
        if sampler:
            sampler.start()
        if profile:
            _lib.check(_lib.lib().ce_dit_profile_begin(model._handle, 1200 * steps))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        prof = None
        if profile:
            import ctypes
            ms = (ctypes.c_double * 4)(); work = (ctypes.c_double * 4)(); cnt = (ctypes.c_int64 * 4)()
            _lib.check(_lib.lib().ce_dit_profile_end(model._handle, ms, work, cnt))
            prof = {"ms": list(ms), "work": list(work), "count": list(cnt)}
        clocks = sampler.stop() if sampler else None
        barrier()
        dev_ms = e0.elapsed_time(e1)
        t = torch.tensor([dev_ms, wall * 1000.0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), prof, clocks

    sampler = ClockSampler(local) if rank == 0 else None
    # pass 1 -- `value`: no per-launch events.  The context cache is emptied right before the timed region, so the timed steps are
    # the FIRST `steps` steps of an edit (the step-invariant context is computed inside the timed region, once).
    for i in range(args.warmup):
        device_step(i)
    model.clear_context_cache()
    launch_count = {"n": 0}
    _orig = device_step

    def counted_step(i):
        _orig(i)
        launch_count["n"] += model.launches_per_forward() + 1   # + the fused sampler launch

    if args.cuda_graph:   # replay the forward as one CUDA graph in the `value` pass (captured during warm-up: step 2 of a configuration)
        model.use_cuda_graph = True
        for i in range(2):
            device_step(args.warmup + i)
        model.clear_context_cache()
    dev_ms, wall_ms, _, clocks = timed(counted_step, args.steps, 0, sampler, profile=False)
    if args.dump_outputs and rank == 0:   # before the passes below overwrite the model's output buffer and the latents
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, v in last.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), v.float().cpu().numpy())
    model.use_cuda_graph = False
    launches = launch_count["n"]
    value = world * args.steps / (dev_ms / 1000.0)
    # pass 2 -- the per-class split (CUDA events around every launch; slightly slower, not the reported value)
    split_steps = min(args.steps, 6)
    split_ms, _, prof, _ = timed(device_step, split_steps, 1, None, profile=True)
    # pass 3 -- e2e through the host-buffer call, same step count as pass 1
    e2e_steps = args.steps
    model.clear_context_cache()
    e2e_dev_ms, e2e_wall_ms, _, _ = timed(host_step, e2e_steps, 2)
    e2e_value = world * e2e_steps / (e2e_wall_ms / 1000.0)
    # pass 4 -- the same loop without the context cache (what round 1 measured), for the record
    nocache_ms = None
    if not args.no_context_cache and rank == 0 and world == 1:
        model.cache_context = False
        model.clear_context_cache()
        nocache_ms, _, _, _ = timed(device_step, min(args.steps, 4), 1)
        nocache_ms /= min(args.steps, 4)
        model.cache_context = True

    # the VAE bookends of one edit (encode of the condition video, decode of the result), timed once per run
    edit = None
    if not args.no_vae:
        vae = ce.AutoencoderKLWan(device=dev)
        gv = torch.Generator(device=dev).manual_seed(7)
        for n, p in vae.named_parameters():
            if n.endswith("gamma"):
                p.data.normal_(0, 0.1, generator=gv).add_(1.0)
            elif n.endswith("bias"):
                p.data.normal_(0, 0.02, generator=gv)
            else:
                fan_in = p[0].numel()
                p.data.normal_(0, 1.0 / fan_in ** 0.5, generator=gv)
        video = torch.zeros(1, 3, 5, 8 * LAT_H, 8 * LAT_W, dtype=torch.bfloat16, device=dev)
        video[:, :, 0] = torch.rand(1, 3, 8 * LAT_H, 8 * LAT_W, device=dev) * 2 - 1
        zlat = torch.randn(1, 16, FRAMES, LAT_H, LAT_W, dtype=torch.bfloat16, device=dev)

        def time_once(fn, reps=2):
            fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        enc_ms = time_once(lambda: vae.encode(video))
        enc_launches = vae.launches()
        dec_ms = time_once(lambda: vae.decode(zlat))
        dec_launches = vae.launches()
        step_ms = dev_ms / args.steps
        edit = {
            "vae_encode_ms": enc_ms, "vae_decode_ms": dec_ms, "vae_encode_launches": enc_launches, "vae_decode_launches": dec_launches,
            "vae_encode_conv_tflops": VAE_ENCODE_FLOP / enc_ms / 1e9,
            "vae_decode_conv_tflops": VAE_DECODE_FLOP / dec_ms / 1e9,
            "vae_decode_algorithmic_GBps": 23.64e9 / dec_ms / 1e6,
            "edits_per_sec_50_steps_all_gpus": world / ((enc_ms + dec_ms + 50 * step_ms) / 1000.0),
            "edits_per_sec_8_steps_no_cfg_all_gpus": world / ((enc_ms + dec_ms + 8 * step_ms / 2) / 1000.0),
            "note": "edit = VAE encode + N denoising steps + VAE decode (SURVEY 8d); text/image encoders excluded ('next' row)",
        }
        del vae
        torch.cuda.empty_cache()

    # library bar (SURVEY 8d "reference GPU path"): the oracle's functional restatement of the reference evaluated by torch eager on
    # this GPU in the reference's bf16 configuration = cuBLAS GEMMs + SDPA (cuDNN fused attention as the reference's own dispatch
    # picks on cc 10.0, chronoedit/_src/modules/attention.py:129-138) + ATen elementwise, same weights, same step (2 forwards + CFG
    # + scheduler glue in torch).  A reported bar next to `value`, timed with CUDA events; not part of any timed region above.
    library_bar = None
    if rank == 0 and world == 1 and not args.no_library_bar:
        try:
            library_bar = library_bar_step_rate(model, d_in, d_text, d_img, dev, args.layers)
        except Exception as e:  # noqa: BLE001
            library_bar = {"error": str(e)[:200]}

    if rank == 0:
        peak_tf, peak_hbm, peak_src = peaks()
        flops_fwd = dit_flops_per_forward(args.layers, FRAMES, LAT_H, LAT_W, TEXT_LEN, 257, batch=2)
        gemm_tf = prof["work"][0] / (prof["ms"][0] / 1000.0) / 1e12 if prof["ms"][0] > 0 else 0.0
        attn_tf = prof["work"][1] / (prof["ms"][1] / 1000.0) / 1e12 if prof["ms"][1] > 0 else 0.0
        kernel_ms = sum(prof["ms"])
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {
                "workload": ("configs[1]: ChronoEdit-14B single edit, 720x1280, 5 px frames -> latent [1,36,2,90,160] (7200 tokens), "
                             "512 text + 257 image tokens, CFG 5.0 (2 forwards/step as one batch-2 call), per-GPU independent edits")
                if FRAMES == 2 else
                ("DEV (not the headline workload): configs[2] temporal-reasoning geometry, 29 px frames -> latent [1,36,8,90,160] "
                 "(28800 tokens), CFG 5.0"),
                "layers": args.layers, "global_batch_edits": world, "parallelism": f"dp{world}",
                "l2": "inputs larger than L2 (32.8 GB of weights stream every forward); no explicit flush",
                "latent_update": ("value and e2e: fused CFG + FlowUniPC step (+ next model input) in one launch (ce_unipc_step); e2e feeds the "
                                  "DiT through ce_dit_forward_host_ex from pinned host buffers every step and reads sample + new latents back"),
                "context_cache": (not args.no_context_cache),
                "context_cache_note": ("step-invariant text/image embedders + cross-attention K/V of all blocks kept across the steps of an edit "
                                       "(ce_dit_forward_ex; bit-identical, tests/test_gpu_baseline_sizes.py); the cache is emptied right before the "
                                       "timed region, so the timed steps are the first steps of an edit and include computing it once; algorithmic "
                                       "FLOPs below stay un-hoisted (222.43 TFLOP/forward)"),
                "ms_per_step_without_context_cache": nocache_ms,
                "cuda_graph": bool(args.cuda_graph),
                "timing": "value: CUDA events around the K steps, no per-launch events; roofline split: separate pass with an event pair per launch",
            },
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_wall_ms / e2e_steps},
            "gpu_launches": launches,
            "roofline": {
                "bound": "tensor", "kernel": "gemm_bf16_2cta_kernel / gemm_bf16_kernel (tcgen05, all Linear layers)",
                "achieved": gemm_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf, "peak_source": peak_src + " bf16_tflops_sustained",
                # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures, as summarised
                # into profiles/traffic.json by scripts/summarize_profiles.py (null when that file has no entry for the kernel)
                "traffic": traffic("gemm"), "traffic_launch": traffic("gemm", "launch"),
                "algorithmic_bytes_of_that_launch": traffic("gemm", "algorithmic_bytes"),
                "launches": prof["count"][0], "ms_total": prof["ms"][0], "split_pass_steps": split_steps, "split_pass_ms_per_step": split_ms / split_steps,
                "share_of_kernel_time": prof["ms"][0] / kernel_ms if kernel_ms else None,
                "attention": {"achieved": attn_tf, "frac": attn_tf / peak_tf, "ms_total": prof["ms"][1], "launches": prof["count"][1],
                              "traffic": traffic("attention"), "traffic_launch": traffic("attention", "launch"),
                              "algorithmic_bytes_of_that_launch": traffic("attention", "algorithmic_bytes")},
                "conv": {"traffic": traffic("conv"), "traffic_launch": traffic("conv", "launch"),
                         "algorithmic_bytes_of_that_launch": traffic("conv", "algorithmic_bytes")},
                "rows_ms_total": prof["ms"][2], "other_ms_total": prof["ms"][3],
                "whole_step": {"algorithmic_tflop_per_step": flops_fwd / 1e12, "achieved": flops_fwd / 1e12 / (dev_ms / args.steps / 1000.0),
                               "frac": flops_fwd / 1e12 / (dev_ms / args.steps / 1000.0) / peak_tf},
            },
            "clocks": clocks,
            "weight_broadcast": {"bytes": bcast_bytes, "seconds_incl_init": round(t_bcast, 3)},
            "edit": edit,
        }
        line["library_bar"] = library_bar
        if world == 1 and not args.no_cpu_baseline:
            rate, times, cores, desc = cpu_reference_step_rate(reps=2, warmup=1)
            line["cpu_baseline"] = {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc,
                                    "extrapolated": "x80 identical blocks only (full token count measured)"}
            try:
                line["cpu_baseline"].update(cpu_extras(cores))
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"]["extras_error"] = str(e)[:200]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=40, help="DEV ONLY: fewer layers make the number invalid as a bench value")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--cuda-graph", action="store_true", help="replay the DiT forward as a CUDA graph in the value pass (A/B)")
    ap.add_argument("--no-context-cache", action="store_true", help="recompute the step-invariant context every step (round-1 behaviour)")
    ap.add_argument("--no-vae", action="store_true", help="skip the (untimed-region) VAE encode/decode measurement")
    ap.add_argument("--latent-frames", type=int, default=2, choices=[2, 8],
                    help="DEV ONLY: 8 = the temporal-reasoning geometry of configs[2] (28 800 tokens); not the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's DiT output and new latents to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
    if args.latent_frames != 2:
        global FRAMES
        FRAMES = args.latent_frames
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
