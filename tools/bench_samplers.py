"""Step count vs cost: DDIM at 200 steps against DPM-Solver++ 2M at 10 / 20 / 25 / 50 steps, at the benchmark shape.

    python tools/bench_samplers.py [--batch 8] [--reps 3] [--out profiles/samplers.json]

Tango base UNet (seeded synthetic weights), `--batch` prompts with CFG 3 (UNet batch 2 x batch), 256 x 16 latents
(10.24 s clips), bf16, 64 synthetic T5 tokens, same seeded initial latents for every run. The configurations are run
in turn, `--reps` rounds, after one warm-up call each (CUDA-graph capture, time-embedding table). For each:
  * per-step time: device events around the denoising loop (AudioDiffusion.last_step_ms), median over the rounds;
  * whole call: inference + VAE decoder + HiFi-GAN to int16, device events around it, as audio seconds per second;
and once, standalone at the same shape: tng_sched_step (the DDIM update) and tng_sched_multistep (orders 1 / 2 / 3),
CUDA events over `--launches` back-to-back launches, with the algorithmic bytes each moves (tango_b200.lib) over that
time. Every DPM run's final latents are compared (printed, not asserted) with a DPM-Solver++ 3M / 200-step run on the
same seeds; no statement about audio quality follows from that distance on random weights.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import statistics

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tango_b200 import lib as L  # noqa: E402
from tango_b200 import synth  # noqa: E402
from tango_b200.pipeline import Tango  # noqa: E402
from tango_b200.schedulers import DDIMScheduler, DPMSolverMultistepScheduler  # noqa: E402

AUDIO_S = (4 * 256 * 160 + 32) / 16000.0


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        return r.stdout.strip()
    except OSError:
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def kernel_times(dev, B, n_launch):
    """Standalone tng_sched_step vs tng_sched_multistep at the loop's shape (CFG, bf16 next input, in-place sample)."""
    Cc, HW = 8, 256 * 16
    g = torch.Generator(device=dev).manual_seed(0)
    mo = torch.randn(2 * B * HW, Cc, device=dev, generator=g)
    sample = torch.randn(B, Cc, 256, 16, device=dev, generator=g)
    ring = [torch.randn(B, Cc, 256, 16, device=dev, generator=g) for _ in range(3)]
    x_in = torch.empty(2 * B * HW, Cc, device=dev, dtype=torch.bfloat16)
    ddim = DDIMScheduler.from_pretrained(None)
    ddim.set_timesteps(200, device=dev)
    dpm = DPMSolverMultistepScheduler.from_pretrained(None, solver_order=3)
    dpm.set_timesteps(20, device=dev)
    c_ddim, c_dpm = ddim.coefficient_table(dev)[5], dpm.coefficient_table(dev)[5]
    runs = {"sched_step (DDIM)": lambda: L.sched_step(mo, True, 3.0, sample, None, c_ddim, sample, x_in, B=B, Cc=Cc,
                                                      HW=HW)}
    for order in (1, 2, 3):
        runs[f"sched_multistep order {order}"] = (lambda o=order: L.sched_multistep(
            mo, True, 3.0, sample, ring[0], ring[1], c_dpm, o, ring[2], sample, x_in, B=B, Cc=Cc, HW=HW))
    out = {}
    for name, fn in runs.items():
        L.PROF.start()
        fn()
        fam = L.PROF.stop()
        nbytes = sum(v["bytes"] for v in fam.values())
        for _ in range(20):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_launch):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / n_launch
        out[name] = {"us": round(us, 3), "algorithmic_bytes": int(nbytes), "gb_s": round(nbytes / us / 1e3, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=2000)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_samplers.py needs a CUDA device")
    torch.set_grad_enabled(False)
    dev = torch.device("cuda:0")
    B = args.batch
    info = card()
    print(f"card: {info}", flush=True)
    cfg = synth.BASE_UNET_CONFIG
    t = Tango.from_synthetic(unet_config=cfg, device=dev, precision="bf16")
    embeds, mask = synth.synth_conditioning(B, 64, cfg["cross_attention_dim"], seed=1)
    embeds, mask = embeds.to(dev), mask.to(dev)
    prompts = [f"synthetic prompt {i}" for i in range(B)]
    runs = [("DDIM", 200, lambda: DDIMScheduler.from_pretrained(None))]
    runs += [("DPM-Solver++ 2M", n, lambda: DPMSolverMultistepScheduler.from_pretrained(None)) for n in (10, 20, 25, 50)]

    def call(sch, steps):
        gen = torch.Generator(device=dev).manual_seed(1234)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lat = t.model.inference(prompts, sch, steps, 3.0, prompt_embeds=embeds, boolean_prompt_mask=mask,
                                generator=gen, latent_shape=(256, 16))
        Bq, Cl, H, W = lat.shape
        t.vae.decode_rows_to_waveform(lat.permute(0, 2, 3, 1).reshape(Bq * H * W, Cl).contiguous(), Bq, H, W)
        e1.record()
        torch.cuda.synchronize()
        return lat.clone(), t.model.last_step_ms, e0.elapsed_time(e1)

    scheds = {(name, n): mk() for name, n, mk in runs}
    for (name, n), sch in scheds.items():          # warm-up: graph capture, time-embedding tables
        call(sch, n)
    res = {k: {"step_ms": [], "call_ms": []} for k in scheds}
    lats = {}
    for _ in range(args.reps):                     # alternate the configurations
        for (name, n), sch in scheds.items():
            lat, step_ms, call_ms = call(sch, n)
            res[(name, n)]["step_ms"].append(step_ms)
            res[(name, n)]["call_ms"].append(call_ms)
            lats[(name, n)] = lat
    ref, _, _ = call(DPMSolverMultistepScheduler.from_pretrained(None, solver_order=3), 200)
    rows = []
    print(f"batch {B} x CFG 3 (UNet batch {2 * B}), 256 x 16 latents ({AUDIO_S:.2f} s clips), bf16, base UNet; "
          f"median of {args.reps} alternating rounds", flush=True)
    for (name, n), r in res.items():
        step = statistics.median(r["step_ms"])
        call_ms = statistics.median(r["call_ms"])
        d = float((lats[(name, n)] - ref).double().norm() / ref.double().norm())
        row = {"sampler": name, "steps": n, "step_ms": round(step, 3), "call_ms": round(call_ms, 1),
               "audio_s_per_s": round(B * AUDIO_S / (call_ms / 1e3), 2),
               "step_ms_all": [round(x, 3) for x in r["step_ms"]], "call_ms_all": [round(x, 1) for x in r["call_ms"]],
               "latent_rel_dist_vs_dpm3m_200": round(d, 4)}
        rows.append(row)
        print(f"  {name:16s} {n:4d} steps: {step:7.3f} ms/step, call {call_ms:8.1f} ms -> {row['audio_s_per_s']:7.2f} "
              f"audio-s/s; latents rel. distance from DPM-Solver++ 3M x 200: {d:.4f}", flush=True)
    kt = kernel_times(dev, B, args.launches)
    print(f"standalone update kernels at B={B}, C=8, HW=4096, CFG, bf16 next input ({args.launches} launches):")
    for k, v in kt.items():
        print(f"  {k:28s} {v['us']:8.3f} us  {v['algorithmic_bytes'] / 1e6:6.2f} MB  {v['gb_s']:7.1f} GB/s")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": info, "batch": B, "reps": args.reps, "runs": rows, "kernels": kt}, f, indent=1)


if __name__ == "__main__":
    main()
