#!/usr/bin/env python
"""Headline benchmark: DADD patient-conditioned progression (13 MES levels x 50 DDIM steps, lambda = 3, 256x256).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--patients P] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one progression batch per GPU: P patients x 13 levels go through conditioning (AOE + purifier), 50
CUDA-graph-replayed denoising steps (UNet + fused DDIM) and the VAE decode, producing P*13 images of 256x256.
Prints ONE JSON line (rank 0).  ``value``: images/s with inputs resident in HBM, timed with CUDA events over exactly K
steps (max over ranks).  ``e2e``: the same through the public API ``sample_progressions`` with pinned HOST inputs - the
patients' CLIP-preprocessed structure images, encoded by the CLIP ViT-L/14 + resampler front end inside the call - and a
device->host read of the finished images inside the timed region.  ``--impl reference`` times the reference's CPU path
(the oracle port: same graph, PyTorch eager fp32 - diffusers is not installable here) on the box's host cores.

After the headline the same run adds (each a separate object of the JSON line):
``parity``   eps max relative error (B = 13, t = 999) and decoded-image PSNR of a 2-level x 50-step progression against the
             CPU oracle, at the dtype the benchmark ran in (north-star gates: 2e-2 / 40 dB);
``strong``   BASELINE config 2 read as STRONG scaling: 8 patients x 13 levels = 104 units in total, split over the ranks;
``config4``  one guidance scale of the evaluation sweep (50 samples x 4 MES classes = 200 jobs, 50 steps) through
             ``evaluation_pipeline.generate_all``, jobs sharded over the ranks;
``config5``  the 512x512 stress progression, batch 16 in total split over the ranks;
``config3``  the training step (batch 8 per GPU, bf16, 256x256: frozen VAE encode + CLIP, conditioning, UNet forward /
             backward, bucketed gradient all-reduce over NCCL, clip + AdamW), with the all-reduce's exposed share.

``--steps K`` is the number of timed repetitions of every leg: the headline, ``e2e``, ``strong``, ``config4`` (sweeps),
``config5`` and ``config3`` (training steps); the kernel rooflines time 20 launches each.

``--dump-outputs DIR`` (rank 0) writes what the last timed step returned: ``DIR/images.npy`` (resident inputs) and
``DIR/e2e_images.npy`` (``sample_progressions``), fp32 (k, 3, 256, 256), the same seeded choice of k images of the batch in
both, k as large as fits ``DUMP_BYTES`` in all; with ``--impl reference``, ``DIR/eps.npy`` (13, 4, 32, 32) of the last timed
UNet step and ``DIR/images.npy`` (13, 3, 256, 256) of the timed decode.  Weights and inputs are seeded, and the convolutions
use cuDNN's heuristic algorithm choice (see ``main``), so two builds run with the same arguments can be compared output for
output.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVELS, DDIM_STEPS, STEER = 13, 50, 3.0
WORKLOAD = ("13 MES levels x 50 DDIM steps, lambda=3, 256x256, SD-1.x-shaped random-init weights, CFG off (routing gates), "
            "eta=0, VAE decode included")
UNET_GFLOP_PER_SAMPLE_STEP = 178.7          # SURVEY.md Appendix C.1
SELF_ATTN_N, SELF_ATTN_D, SELF_ATTN_H = 1024, 40, 8
DUMP_BYTES = 64_000_000


_RESULT_FD = None      # the process's original stdout: carries exactly one JSON line


def _claim_stdout() -> None:
    """Point fd 1 at stderr for the rest of the run (library banners such as NCCL's version line are written straight to fd 1)
    and keep the original stdout for the result line."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def _emit(result: dict) -> None:
    line = (json.dumps(result) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of ``kernel`` at the bench batch, from the committed
    ``ncu --set full`` capture summarised in profiles/ncu_traffic.json (None when that kernel has no capture yet)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[kernel]["bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------- CPU reference
def cpu_reference_sample(batch: int, seed: int = 0):
    """A bounded sample of the reference CPU path: ONE UNet denoising step at B = 13 (of the 50) through the oracle
    port, plus ONE VAE decode at B = 13; returns (unet_step, decode, cores, last): the two timed callables return seconds and
    leave what they computed in ``last`` ("eps", "images")."""
    import torch
    from oracle import conditioning, unet as ounet, weights
    torch.set_num_threads(os.cpu_count() or 1)
    state = weights.make_module_state(seed=seed)
    uw, aw, pw, vw = (weights.sub_state(state, p) for p in ("unet.unet.", "ordinal_embedder.", "feature_purifier.", "vae.vae."))
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 4, 32, 32, generator=g).repeat(batch, 1, 1, 1)
    img = torch.randn(1, 16, 768, generator=g).expand(batch, -1, -1).contiguous()
    tgt, src = torch.linspace(0, 3, batch), torch.zeros(batch)
    t = torch.full((batch,), 999, dtype=torch.long)
    last = {}
    with torch.no_grad():
        cond = conditioning.prepare_conditioning(aw, pw, tgt, src, img)

        def unet_step():
            t0 = time.perf_counter()
            last["eps"] = ounet.unet_forward(uw, x, t, cond, ounet.CrossCfg(True, STEER))
            return time.perf_counter() - t0

        def decode():
            t0 = time.perf_counter()
            last["images"] = ounet.latents_to_images(vw, x)
            return time.perf_counter() - t0
        return unet_step, decode, torch.get_num_threads(), last


def run_reference(args) -> None:
    """The reference's CPU path on the box's host cores.  One timed "step" = ONE UNet denoising step of one patient's 13-level
    progression (B = 13) - a bounded sample of the 50 a progression takes; ``value`` scales it to the whole progression
    (50 x mean step + one timed VAE decode) and ``ms_per_step`` is the timed unit itself."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    unet_step, decode, cores, last = cpu_reference_sample(LEVELS)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):               # untimed passes (each is ~1 s of host work)
            unet_step()
        t_unet = [unet_step() for _ in range(args.steps)]
        t_dec = decode()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    per_step = statistics.mean(t_unet)
    progression_s = DDIM_STEPS * per_step + t_dec
    value = LEVELS / progression_s
    sample = (f"{args.steps} timed UNet denoising step(s) at B=13 (oracle port, fp32 eager, {cores} threads), mean {per_step * 1e3:.0f} ms, "
              f"+ 1 VAE decode at B=13 ({t_dec:.2f} s); one 13x50 progression = 50 x step + decode = {progression_s:.1f} s")
    _emit({
        "impl": "reference", "metric": "progression img/s (13 MES x 50 DDIM steps)", "value": value, "unit": "img/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
        "step_unit": "one UNet denoising step at B=13 (1/50 of a progression); value = 13 / (50 x step + decode)",
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "patients_per_gpu": args.patients, "levels": LEVELS, "ddim_steps": DDIM_STEPS,
                   "images_per_step_per_gpu": args.patients * LEVELS,
                   "note": "the CPU arm times one patient (13 images) at a time; img/s does not depend on how many patients queue"},
        "cpu_baseline": {"value": value, "unit": "img/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def parity_block(dev, cdt) -> dict:
    """North-star gates measured in this run at the benchmark's dtype, product vs the CPU oracle (the checker, never the thing
    timed): eps max relative error for one patient's 13 levels at t = 999, and decoded-image PSNR after a 2-level x 50-step
    progression (same weights, noise and conditioning on both sides)."""
    import math
    import torch
    import progressive_stable_diffusion_b200 as P
    from oracle import conditioning, sampler, unet as ounet, weights
    from progressive_stable_diffusion_b200.inference_pipeline_ip import (_ddim_sample_ip, _latents_to_images, _prepare_conditioning,
                                                                         _set_delta_scale_on_processors)
    torch.set_num_threads(os.cpu_count() or 1)
    state = weights.make_module_state(seed=0)
    module = P.DiffusionModuleWithIP(P.default_config())
    module.load_state_dict(state, strict=True)
    module.to(dev).eval()
    uw, aw, pw, vw = (weights.sub_state(state, p) for p in ("unet.unet.", "ordinal_embedder.", "feature_purifier.", "vae.vae."))
    g = torch.Generator().manual_seed(7)
    noise = torch.randn(1, 4, 32, 32, generator=g)
    tok1 = torch.randn(1, 16, 768, generator=g)
    rel = lambda a, r: ((a.double().cpu() - r.double()).abs().max() / r.double().abs().max()).item()
    with torch.no_grad():
        # eps: one patient's 13 levels, first sampler position
        tgt, src = torch.linspace(0, 3, LEVELS), torch.zeros(LEVELS)
        tok = tok1.expand(LEVELS, -1, -1).contiguous()
        x, t = noise.repeat(LEVELS, 1, 1, 1), torch.full((LEVELS,), 999, dtype=torch.long)
        cond_ref = conditioning.prepare_conditioning(aw, pw, tgt, src, tok)
        eps_ref = ounet.unet_forward(uw, x, t, cond_ref, ounet.CrossCfg(True, STEER))
        cond = _prepare_conditioning(module, tgt.to(dev), src.to(dev), tok.to(dev))
        _set_delta_scale_on_processors(module, STEER)
        eps_err = rel(module(x.to(dev), t.to(dev), cond), eps_ref)
        # images: 2 levels x 50 steps
        tgt2, src2, tok2 = torch.tensor([0.75, 3.0]), torch.ones(2), tok1.expand(2, -1, -1).contiguous()
        lat_ref = sampler.ddim_sample(uw, aw, pw, tgt2, src2, tok2, noise, sampling_steps=DDIM_STEPS, steer_scale=STEER)
        img_ref = ounet.latents_to_images(vw, lat_ref)
        lat = _ddim_sample_ip(module, tgt2, src2, tok2.to(dev), DDIM_STEPS, dev, steer_scale=STEER, init_latents=noise)
        psnr = lambda a: (lambda mse: 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse))(((a.double().cpu() - img_ref.double()) ** 2).mean().item())
        p_full, p_lat = psnr(_latents_to_images(module, lat)), psnr(ounet.latents_to_images(vw, lat.cpu()))
    del module
    torch.cuda.empty_cache()
    return {"dtype": str(cdt).replace("torch.", ""), "eps_max_rel_err": eps_err, "eps_gate": 2e-2, "psnr_db": p_full,
            "psnr_db_oracle_decoder": p_lat, "psnr_gate_db": 40.0, "latent_max_rel_err_50_steps": rel(lat, lat_ref),
            "pass": bool(eps_err <= 2e-2 and p_full >= 40.0 and p_lat >= 40.0),
            "how": "product (CUDA path, this dtype) vs oracle port (CPU fp32), same seeded weights / noise / tokens: eps at B=13, "
                   "t=999, lambda=3; PSNR of the decoded images of a 2-level x 50-step progression (product decoder, and the "
                   "oracle decoder on the product latents)"}


# --------------------------------------------------------------------------------------------------- B200 arm
def dump_outputs(out_dir: str, arrays: dict) -> None:
    """``out_dir/<name>.npy`` for each tensor of ``arrays`` (all with the same leading batch dimension): fp32, the same seeded
    choice of batch entries from each, as many as fit ``DUMP_BYTES`` in all."""
    import numpy as np
    import torch
    batch = next(iter(arrays.values())).shape[0]
    k = min(batch, DUMP_BYTES // sum(t[0].numel() * 4 for t in arrays.values()))
    pick = torch.randperm(batch, generator=torch.Generator().manual_seed(0))[:k].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[pick.to(t.device)].float().cpu().numpy())


def run_b200(args) -> None:
    import torch
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import _lib, ops, parallel
    from progressive_stable_diffusion_b200.inference_pipeline_ip import (_latents_to_images, _sample, _build_labels,
                                                                         sample_progressions)

    rank, local, world = parallel.init_from_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pk = peaks()
    patients, batch = args.patients, args.patients * LEVELS
    cdt = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    P.set_compute_dtype(cdt)

    torch.manual_seed(0)                                          # random-init SD-1.x-shaped weights (PyTorch default inits)
    module = P.DiffusionModuleWithIP(P.default_config(), build_image_encoder=True, build_vae_encoder=True)     # + random-init CLIP ViT-L/14 + resampler, VAE encoder (training leg)
    module.to(dev).eval()

    g = torch.Generator().manual_seed(100 + rank)
    host_tokens = torch.randn(patients, 16, 768, generator=g).pin_memory()
    host_pixels = torch.randn(patients, 3, 224, 224, generator=g).pin_memory()      # CLIP-preprocessed structure images
    host_source = torch.zeros(patients).pin_memory()
    host_noise = torch.randn(patients, 4, 32, 32, generator=g).pin_memory()
    host_images = torch.empty(batch, 3, 256, 256, dtype=torch.float32).pin_memory()
    d_tokens = host_tokens.to(dev).repeat_interleave(LEVELS, 0)
    d_source = host_source.to(dev).repeat_interleave(LEVELS)
    d_target = _build_labels(LEVELS, 0.0, 3.0, dev).repeat(patients)
    d_noise = host_noise.to(dev).repeat_interleave(LEVELS, 0)

    last = {}

    def step_resident():
        lat = _sample(module, d_target, d_source, d_tokens, d_noise, DDIM_STEPS, dev, 0.0, 1.0, None, STEER, 1.0, False, True)
        last["images"] = _latents_to_images(module, lat)

    def step_e2e():
        imgs = sample_progressions(module, host_pixels, host_source, LEVELS, DDIM_STEPS, dev, steer_scale=STEER,
                                   init_latents=host_noise)
        host_images.copy_(imgs, non_blocking=True)

    def timed(fn, steps):
        parallel.barrier()
        torch.cuda.synchronize(dev)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(steps):
            fn()
        end.record()
        torch.cuda.synchronize(dev)
        parallel.barrier()
        return parallel.max_over_ranks(start.elapsed_time(end) / 1e3, dev)

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step_resident()
        step_e2e()
        torch.cuda.synchronize(dev)
        eng = next(iter(module.__dict__["_b200_engines"].values()))
        sampler = ClockSampler(local).start() if rank == 0 else None
        _lib.reset_launch_count()
        seconds = timed(step_resident, args.steps)
        eager_launches = _lib.launch_count()
        images_resident = last.pop("images")
        seconds_e2e = timed(step_e2e, args.steps)
        clocks = sampler.stop() if sampler else None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"images": images_resident, "e2e_images": host_images})
        del images_resident

        # ---- dominant kernel, timed live on the launching stream: self-attention N=1024, d=40 at this batch (a kernel timed
        # alone, after a pause that lets the power-capped clocks of the long step recover: the burst peaks are its roofline) ----
        time.sleep(3.0)
        c = SELF_ATTN_H * SELF_ATTN_D
        qkv = torch.randn(batch, SELF_ATTN_N, 3 * c, device=dev, dtype=cdt)
        reps = 20
        for _ in range(3):
            ops.self_attention(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], SELF_ATTN_H)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            ops.self_attention(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], SELF_ATTN_H)
        e1.record()
        torch.cuda.synchronize(dev)
        attn_s = e0.elapsed_time(e1) / 1e3 / reps
        attn_flop = 4.0 * SELF_ATTN_N * SELF_ATTN_N * c * batch
        # ---- GroupNorm+SiLU 320ch @32x32 (the most frequent memory-bound kernel); a rotation of input/output pairs larger
        # than the 126 MB L2 so that no launch finds its operands cached ----
        nbuf = max(2, -(-(160 << 20) // (batch * 320 * 32 * 32 * 2 * 2)))
        xgs = [torch.randn(batch, 320, 32, 32, device=dev, dtype=cdt).contiguous(memory_format=torch.channels_last)
               for _ in range(nbuf)]
        ygs = [torch.empty_like(x) for x in xgs]
        gam, bet = torch.ones(320, device=dev), torch.zeros(320, device=dev)
        for i in range(nbuf):
            ops.group_norm(xgs[i], gam, bet, 32, 1e-5, True, out=ygs[i])
        torch.cuda.synchronize(dev)
        e0.record()
        for i in range(reps):
            ops.group_norm(xgs[i % nbuf], gam, bet, 32, 1e-5, True, out=ygs[i % nbuf])
        e1.record()
        torch.cuda.synchronize(dev)
        gn_s = e0.elapsed_time(e1) / 1e3 / reps
        gn_bytes = xgs[0].numel() * 2 * 2
        # ---- triple-pathway cross-attention N=1024, d=40 (tcgen05 kernel; HBM-bound: Q in + O out) ----
        qx = [torch.randn(batch, SELF_ATTN_N, c, device=dev, dtype=cdt) for _ in range(3)]
        kc = torch.randn(batch, SELF_ATTN_H, 48, SELF_ATTN_D, device=dev, dtype=cdt)
        vc = torch.randn(batch, SELF_ATTN_H, 48, SELF_ATTN_D, device=dev, dtype=cdt)
        gts = torch.tensor([0.9, 0.1, STEER], device=dev)
        for i in range(3):
            ops.cross_attention(qx[i], kc, vc, gts, SELF_ATTN_H, 16, 3)
        torch.cuda.synchronize(dev)
        e0.record()
        for i in range(reps):
            ops.cross_attention(qx[i % 3], kc, vc, gts, SELF_ATTN_H, 16, 3)
        e1.record()
        torch.cuda.synchronize(dev)
        xa_s = e0.elapsed_time(e1) / 1e3 / reps
        xa_bytes = qx[0].numel() * 2 * 2 + kc.numel() * 2 * 2
        # ---- residual add + LayerNorm N=1024, C=320 (reads x and r, writes the sum and the norm); operands rotate through
        # more than the L2 ----
        lnw, lnb = torch.ones(c, device=dev), torch.zeros(c, device=dev)
        for i in range(3):
            ops.add_layer_norm(qx[i], qx[(i + 1) % 3], lnw, lnb, 1e-5)
        torch.cuda.synchronize(dev)
        e0.record()
        for i in range(reps):
            ops.add_layer_norm(qx[i % 3], qx[(i + 1) % 3], lnw, lnb, 1e-5)
        e1.record()
        torch.cuda.synchronize(dev)
        ln_s = e0.elapsed_time(e1) / 1e3 / reps
        ln_bytes = qx[0].numel() * 2 * 4

        extras = {}
        if not args.no_extras:
            from progressive_stable_diffusion_b200.evaluation_pipeline import generate_all
            # ---- strong scaling of config 2: 8 patients x 13 levels = 104 units IN TOTAL, split over the ranks ----
            sp = 8 // world if 8 % world == 0 else 0                 # patients per rank
            if sp == patients:
                extras["strong"] = {"units_total": 8 * LEVELS, "units_per_gpu": batch, "value": batch * world * args.steps / seconds,
                                    "unit": "img/s", "ms_per_step": seconds / args.steps * 1e3, "note": "identical to the headline run"}
            elif 0 < sp < patients:
                s_tok, s_src = d_tokens[:sp * LEVELS], d_source[:sp * LEVELS]
                s_tgt, s_noise = d_target[:sp * LEVELS], d_noise[:sp * LEVELS]

                def step_strong():
                    lat = _sample(module, s_tgt, s_src, s_tok, s_noise, DDIM_STEPS, dev, 0.0, 1.0, None, STEER, 1.0, False, True)
                    return _latents_to_images(module, lat)
                for _ in range(3):
                    step_strong()
                sec = timed(step_strong, args.steps)
                extras["strong"] = {"units_total": 8 * LEVELS, "units_per_gpu": sp * LEVELS, "value": 8 * LEVELS * args.steps / sec,
                                    "unit": "img/s", "ms_per_step": sec / args.steps * 1e3,
                                    "note": "fixed total work (8 patients x 13 levels) over all ranks; efficiency = value / (N=1 value) / N"}
            # ---- config 4: one guidance scale of the evaluation sweep (50 samples x 4 classes), 50 steps, jobs sharded ----
            n_jobs = 200
            jobs = sorted((i % 16, float(i % 4), float(i // 50)) for i in range(n_jobs))       # (token set, source MES, target MES)
            g4 = torch.Generator().manual_seed(4)
            tok16 = torch.randn(16, 16, 768, generator=g4).to(dev)
            bs4 = -(-n_jobs // world)
            bs4 = min(bs4, 100)

            def step_cfg4():
                return generate_all(module, jobs, tok16, dev, batch_size=bs4, sampling_steps=DDIM_STEPS, steer_scale=STEER,
                                    rank=rank, world_size=world)
            step_cfg4()
            sec = timed(step_cfg4, args.steps) / args.steps
            extras["config4"] = {"workload": "evaluation sweep, ONE of the 5 scales: 50 samples x 4 MES classes = 200 jobs x 50 DDIM steps "
                                             "through generate_all (decode + copy to host included), jobs sharded over the ranks",
                                 "jobs": n_jobs, "batch_per_rank": bs4, "value": n_jobs / sec, "unit": "img/s", "seconds": sec,
                                 "timed_sweeps": args.steps, "full_sweep_estimate_s": 5 * sec}
            # ---- config 5: 512x512 (64x64 latents) progression, 16 units in total ----
            if 16 % world == 0:
                u5 = 16 // world
                t5 = torch.linspace(0.0, 3.0, 16, device=dev)[rank * u5:(rank + 1) * u5].contiguous()
                s5 = torch.zeros(u5, device=dev)
                k5 = d_tokens[:1].expand(u5, -1, -1).contiguous()
                n5 = torch.randn(1, 4, 64, 64, generator=g4).to(dev).expand(u5, -1, -1, -1).contiguous()

                def step_cfg5():
                    lat = _sample(module, t5, s5, k5, n5, DDIM_STEPS, dev, 0.0, 1.0, None, STEER, 1.0, False, True)
                    return _latents_to_images(module, lat)
                module.cfg.dataset.image_size = 512                  # (the sampler engine sizes its latents from the config)
                try:
                    step_cfg5()
                    step_cfg5()
                    sec = timed(step_cfg5, args.steps)
                finally:
                    module.cfg.dataset.image_size = 256
                extras["config5"] = {"workload": "512x512 (64x64x4 latents) progression stress: 16 units x 50 DDIM steps, lambda=3, VAE decode "
                                                 "included; self-attention at N=4096 / 1024 / 256", "units_total": 16, "units_per_gpu": u5,
                                     "value": 16 * args.steps / sec, "unit": "img/s", "ms_per_step": sec / args.steps * 1e3}

    with torch.no_grad():
        if args.profile_step:      # one eager denoising step between cudaProfilerStart/Stop (ncu --profile-from-start off)
            eng.state.zero_()
            eng._step()
            torch.cuda.synchronize(dev)
            eng.state.zero_()
            torch.cuda.profiler.start()
            eng._step()
            torch.cuda.synchronize(dev)
            torch.cuda.profiler.stop()

    if not args.no_extras:
        # ---- config 3: training step, batch 8 per GPU, bf16, DDP gradient all-reduce (LAST: it updates the weights) ----
        from progressive_stable_diffusion_b200 import training as T
        tb = 8
        gt = torch.Generator(device=dev).manual_seed(300 + rank)
        t_images = torch.rand(tb, 3, 256, 256, device=dev, generator=gt) * 2 - 1
        t_struct = torch.randn(tb, 3, 224, 224, device=dev, generator=gt)
        t_labels = torch.randint(0, 4, (tb,), device=dev, generator=gt).float()
        trainer = T.DataParallelTrainer(module, lr=1e-5, weight_decay=0.01, max_grad_norm=1.0)
        step_train = lambda: trainer.step(lambda: T.training_step(module, (t_images, t_labels, t_struct), generator=gt,
                                                                   compute_dtype=torch.bfloat16))
        for _ in range(2):
            step_train()
        _lib.reset_launch_count()
        sec_eager = timed(step_train, args.steps)
        train_launches = _lib.launch_count() // args.steps
        # the whole step (forward, backward, bucket all-reduces, clip, AdamW) as ONE captured graph: the eager step is host-bound
        graphed, why = True, ""
        try:
            replay = trainer.capture(lambda: T.training_step(module, (t_images, t_labels, t_struct), generator=gt,
                                                             compute_dtype=torch.bfloat16), generators=(gt,))
            replay()
            torch.cuda.synchronize(dev)
            sec = timed(replay, args.steps)
        except Exception as e:      # noqa: BLE001 - capture is an optimisation: report and keep the eager number
            graphed, why, sec = False, f"{type(e).__name__}: {e}"[:200], sec_eager
        extras["config3"] = {"workload": "training step, batch 8 per GPU, bf16 compute / fp32 master weights, 256x256: VAE encode + CLIP "
                                         "(frozen), AOE / purifier / resampler, UNet forward + backward, Min-SNR loss, bucketed all-reduce, "
                                         "clip 1.0, AdamW (4 groups)", "batch_per_gpu": tb, "value": tb * world * args.steps / sec, "unit": "img/s",
                             "ms_per_step": sec / args.steps * 1e3, "dadd_launches_per_step": int(train_launches),
                             "grad_buckets": len(trainer.buckets), "grad_bytes": int(sum(bk.numel for bk in trainer.buckets) * 4),
                             "cuda_graph": graphed, "ms_per_step_eager": sec_eager / args.steps * 1e3}
        if why:
            extras["config3"]["cuda_graph_error"] = why
        if world > 1:           # exposed share of the gradient all-reduce: the same step with the collective switched off
            if graphed:
                trainer._skip_allreduce = True
                replay()
                sec_off = timed(replay, args.steps)
                trainer._skip_allreduce = False
            else:
                trainer.world = 1
                step_train()
                sec_off = timed(step_train, args.steps)
                trainer.world = world
            extras["config3"]["ms_per_step_without_allreduce"] = sec_off / args.steps * 1e3
            extras["config3"]["allreduce_exposed_share"] = max(0.0, 1.0 - sec_off / sec)
        del trainer

    images_total = batch * world * args.steps
    value = images_total / seconds
    e2e_value = images_total / seconds_e2e
    launches = eager_launches + args.steps * DDIM_STEPS * eng.launches_per_step
    # every rank leaves the process group BEFORE rank 0 times the CPU baseline: a rank parked in a collective keeps a host
    # thread spinning, and one extra busy thread on a fully subscribed OpenMP team slows the baseline ~10x (measured)
    parallel.barrier()
    parallel.shutdown()
    if rank != 0:
        return
    if hasattr(os, "sched_setaffinity"):          # undo any affinity narrowing inherited from the communication library
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    unet_step, decode, cores, _ = cpu_reference_sample(LEVELS)
    unet_step()
    t_unet, t_dec = unet_step(), decode()
    cpu_progression = DDIM_STEPS * t_unet + t_dec
    if not args.no_extras:
        extras["parity"] = parity_block(dev, cdt)
    tflops = batch * world * args.steps * DDIM_STEPS * UNET_GFLOP_PER_SAMPLE_STEP / 1e3 / seconds
    _emit({
        "metric": "progression img/s (13 MES x 50 DDIM steps)", "value": value, "unit": "img/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": seconds / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": WORKLOAD, "patients_per_gpu": patients, "levels": LEVELS, "ddim_steps": DDIM_STEPS, "images_per_step_per_gpu": batch,
                   "parallelism": f"independent (patient x level) units, {world} rank(s), no data-path collective",
                   "l2": "inputs larger than L2: 1.8 GB of 16-bit weights stream through the 126 MB L2 on every UNet pass"},
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": int(host_pixels.numel() * 4 + host_source.numel() * 4 + host_noise.numel() * 4),
                "path": "sample_progressions(host pixels (P,3,224,224) -> CLIP ViT-L/14 + resampler once per patient -> purifier/AOE -> "
                        "50 graph-replayed steps -> VAE decode) -> pinned host images",
                "d2h_bytes_per_step": int(host_images.numel() * 4), "ms_per_step": seconds_e2e / args.steps * 1e3},
        "gpu_launches": int(launches),
        "dadd_launches_per_denoising_step": int(eng.launches_per_step),
        "unet_tflops_achieved": tflops, "unet_frac_of_sustained_bf16_peak": tflops / pk["bf16_tflops_sustained"] / world,
        "clocks": clocks,
        "roofline": {"kernel": "self_attn (N=1024, d=40, H=8) at the bench batch", "bound": "tensor",
                     "achieved": attn_flop / attn_s / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": attn_flop / attn_s / 1e12 / pk["bf16_tflops"], "traffic": ncu_traffic("self_attn"),
                     "peak_source": pk["source"], "us_per_launch": attn_s * 1e6,
                     "limiter": "MUFU.EX2 (16/clk/SM = one warp instruction per 8 clk per scheduler): 160 flop per exponential at d=40 "
                                "caps the kernel at 744 TFLOP/s = 45 % of the tensor peak; the kernel runs at 9.5 clk per exponential "
                                "(profiles/r02_attn_microbench.txt)"},
        "roofline_groupnorm": {"kernel": "groupnorm+silu NHWC 320ch 32x32 at the bench batch", "bound": "hbm",
                               "achieved": gn_bytes / gn_s / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                               "frac": gn_bytes / gn_s / 1e9 / pk["hbm_gbs"], "traffic": ncu_traffic("groupnorm"),
                               "us_per_launch": gn_s * 1e6},
        "roofline_cross_attn": {"kernel": "triple-pathway cross_attn (N=1024, d=40, 48 tokens) at the bench batch", "bound": "hbm",
                                "achieved": xa_bytes / xa_s / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                "frac": xa_bytes / xa_s / 1e9 / pk["hbm_gbs"], "traffic": ncu_traffic("cross_attn"),
                                "us_per_launch": xa_s * 1e6},
        "roofline_add_layernorm": {"kernel": "residual add + LayerNorm (N=1024, C=320) at the bench batch", "bound": "hbm",
                                   "achieved": ln_bytes / ln_s / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                   "frac": ln_bytes / ln_s / 1e9 / pk["hbm_gbs"], "traffic": ncu_traffic("add_layernorm"), "us_per_launch": ln_s * 1e6},
        "cpu_baseline": {"value": LEVELS / cpu_progression, "unit": "img/s", "cores": cores, "kind": "port",
                         "sample": f"1 UNet denoising step at B=13 ({t_unet:.2f} s) + 1 VAE decode at B=13 ({t_dec:.2f} s) through the "
                                   f"oracle port (fp32 eager); 13x50 progression extrapolated = {cpu_progression:.1f} s"},
        **extras,
    })


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed repetitions of every leg (see above)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--patients", type=int, default=8, help="patient progressions per GPU per step (13 images each)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["bf16", "fp16"],
                    help="16-bit operand type of the kernels.  fp16 (default; the reference's own mixed-precision dtype, "
                         "evaluation_pipeline.py:943) passes every north-star gate; bf16 has the same rate and bytes but lands at "
                         "26-30 dB PSNR after 50 steps on random-init weights (profiles/r01_precision_experiment.txt)")
    ap.add_argument("--no-extras", action="store_true", help="skip the parity / strong / config4 / config5 legs")
    ap.add_argument("--profile-step", action="store_true",
                    help="after the timed region run ONE eager denoising step inside cudaProfilerStart/Stop (for the ncu launch list)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/*.npy (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # torchrun exports OMP_NUM_THREADS=1 to every rank; rank 0 also times the CPU baseline and needs the host's cores (set before
    # torch is imported).
    if int(os.environ.get("RANK", "0")) == 0:
        os.environ["OMP_NUM_THREADS"] = os.environ["MKL_NUM_THREADS"] = str(os.cpu_count() or 1)
    # cuDNN's heuristic convolution algorithms, not the ones it times per process: timed picks differ from run to run, and
    # the rounding differences grow over 50 fp16 denoising steps, so the images of two runs on the same inputs would differ
    os.environ.setdefault("DADD_CUDNN_BENCHMARK", "0")
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
