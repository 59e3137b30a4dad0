#!/usr/bin/env python
"""bench.py — audio-seconds generated per wall-second on the Tango hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic prompts: `denoise_steps` (200) CFG denoising steps
of the Tango base UNet on a batch of 8 prompts (UNet batch 16, 64 synthetic T5 tokens), then the VAE decoder and the
HiFi-GAN vocoder -> 8 x 163 872 int16 samples (10.24 s each). Workload = BASELINE.json configs[1].

Printed JSON (rank 0, one line):
  value      audio-s/s, inputs resident in HBM, device-timed (CUDA events), max over ranks, whole job
  e2e        same metric through the public API (Tango.generate_for_batch) with HOST buffers: pinned-host prompt
             embeddings copied H2D and the int16 waveforms copied D2H inside the timed region
  roofline   dominant kernel (tcgen05 implicit-GEMM conv/linear): algorithmic FLOPs / CUDA-event time per launch
             against the measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline  the oracle port timed on this box's host cores on a bounded sample (N=1 only)
`--impl reference` times the reference's CPU arithmetic (oracle port; the Python reference itself cannot travel to the
GPU box) on the same config / metric.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (latents, float and int16 waveforms) as
DIR/<name>.npy in float32. Inputs, weights and noise are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

AUDIO_S_PER_SAMPLE = 163872 / 16000.0  # 10.242 s (hifigan: 1024 mel frames -> 163 872 samples)
F_UNET, F_VAE, F_VOC = 803.181e9, 670.468e9, 1027.036e9  # SURVEY.md §8d, per sample, FLOP = 2 MAC


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_inputs(B: int, tokens: int, dim: int, rank: int):
    from tango_b200 import synth
    embeds, mask = synth.synth_conditioning(B, tokens, dim, seed=1 + rank)
    return embeds, mask


# ------------------------------------------------------------------------------------------------- reference arm
def host_threads():
    """Fixed rule for the CPU arm (both the in-line cpu_baseline leg and --impl reference): one thread per PHYSICAL core
    this process may run on (oversubscribing SMT siblings makes torch's CPU convolutions slower, not faster)."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or 0
    except Exception:
        phys = 0
    try:
        allowed = len(os.sched_getaffinity(0))
    except Exception:
        allowed = os.cpu_count() or 1
    n = min(phys, allowed) if phys else allowed
    return max(1, n)


class CpuReference:
    """The reference's CPU arithmetic for the path (oracle port, see oracle/__init__.py), MEASURED at the c2 batch:
    one "step" = one denoising step of the benchmark's batch = ONE CFG UNet forward at UNet batch 2 x args.batch
    (16 x 8 x 256 x 16 latents, 64 tokens), fp32, torch CPU; the decode leg = VAE decoder + HiFi-GAN for the whole
    batch. Nothing is extrapolated from a smaller batch; only the number of denoising steps (200, identical cost each)
    is scaled from the measured steps."""

    def __init__(self, args):
        from oracle import hifigan as ohifi
        from oracle import unet as ounet
        from oracle import vae as ovae
        from tango_b200 import synth
        torch.set_grad_enabled(False)
        self.args, self.ounet, self.ovae, self.ohifi, self.synth = args, ounet, ovae, ohifi, synth
        self.cores = host_threads()
        torch.set_num_threads(self.cores)
        self.cfg = synth.BASE_UNET_CONFIG if args.unet == "base" else synth.XL_UNET_CONFIG
        self.usd = synth.synth_state_dict(synth.unet_param_shapes(self.cfg), 0)
        self.vsd = synth.synth_state_dict(synth.vae_decoder_param_shapes(), 0)
        B = args.batch
        self.embeds, self.mask = synthetic_inputs(B, args.tokens, self.cfg["cross_attention_dim"], 0)
        g = torch.Generator().manual_seed(1234)
        self.lat = torch.randn(B, 8, args.latent_h, 16, generator=g)

    def step_seconds(self, i):
        """One denoising step at the benchmark batch: the CFG-doubled UNet forward (models.py:235-243)."""
        x = torch.cat([self.lat] * 2)
        t0 = time.perf_counter()
        self.ounet.unet_forward(self.usd, self.cfg, x, torch.tensor(995 - 5 * (i % 199)), self.embeds, self.mask)
        return time.perf_counter() - t0

    def decode_seconds(self, n=None):
        """decode_first_stage + decode_to_waveform for n samples of the batch (default: all of it), one at a time as
        a memory-bounded CPU run would; returns seconds for the WHOLE batch (n < batch is scaled by batch / n)."""
        B = self.args.batch
        n = B if n is None else max(1, min(n, B))
        t0 = time.perf_counter()
        for k in range(n):
            mel = self.ovae.decode_first_stage(self.vsd, self.lat[k:k + 1], self.synth.VAE_CONFIG["scale_factor"])
            self.ohifi.decode_to_waveform(self.vsd, mel)
        return (time.perf_counter() - t0) * B / n

    def describe(self, t_step, n_steps, t_dec, n_dec):
        a = self.args
        return (f"oracle port, torch CPU fp32, {self.cores} threads (= physical cores): {n_steps} measured denoising step(s) at "
                f"the benchmark batch (UNet batch {2 * a.batch}, {a.latent_h}x16 latents, {a.tokens} tokens) = {t_step:.2f} s "
                f"each; VAE+HiFi-GAN measured on {n_dec} of {a.batch} samples = {t_dec:.2f} s per batch; "
                f"pass = {a.denoise_steps} x step + decode")


def run_reference(args):
    """`--impl reference`: the reference's CPU arithmetic for this path on the box's host cores (rank 0 only). The
    requested K timed steps are capped so that the run ends within a few minutes (each step costs tens of seconds at the
    c2 batch): `steps_timed` says how many were actually timed; warm-up is one step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_start = time.perf_counter()
    ref = CpuReference(args)
    ref.step_seconds(0)                                    # warm-up (allocator, thread pool)
    times = []
    budget_s = args.reference_budget_s
    while len(times) < max(1, args.steps):
        times.append(ref.step_seconds(len(times) + 1))
        if len(times) >= 2 and time.perf_counter() - t_start + times[-1] > budget_s:
            break
    t_step = float(np.mean(times))
    n_dec = args.batch if t_step * 0.6 * args.batch < 60 else 2
    t_dec = ref.decode_seconds(n_dec)
    per_pass = args.denoise_steps * t_step + t_dec
    audio_s = (4 * args.latent_h * 160 + 32) / 16000.0
    value = args.batch * audio_s / per_pass
    line = {"impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_timed": len(times), "warmup_timed": 1,
            "ms_per_step": per_pass * 1e3, "timed_region_s": float(np.sum(times)) + t_dec * n_dec / args.batch,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, 1),
            "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": ref.cores, "kind": "port",
                             "sample": ref.describe(t_step, len(times), t_dec, n_dec),
                             "step_s": times, "decode_s_per_batch": t_dec},
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": "Tango " + args.unet + " UNet, batch %d prompts/GPU x %d GPU, %d %s steps, "
                        "CFG %.1f, %.2f s clips, 64 synthetic T5 tokens, + VAE decoder + HiFi-GAN -> int16 16 kHz"
                        % (args.batch, world, args.denoise_steps, args.scheduler.upper(), args.guidance,
                           (4 * args.latent_h * 160 + 32) / 16000.0),
            "global_batch": args.batch * world, "unet_batch_per_gpu": 2 * args.batch, "denoise_steps": args.denoise_steps,
            "scheduler": args.scheduler, "guidance": args.guidance, "precision": args.precision,
            "parallelism": f"prompt-shard x{world}", "l2": "working set (1.7 GB bf16 weights + activations) >> 126 MB L2"}


# ------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    from tango_b200 import lib as L
    from tango_b200 import parallel, synth
    from tango_b200.pipeline import Tango
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)

    cfg = synth.BASE_UNET_CONFIG if args.unet == "base" else synth.XL_UNET_CONFIG
    B = args.batch
    latent_shape = (args.latent_h, 16)
    audio_s = (4 * args.latent_h * 160 + 32) / 16000.0   # HiFi-GAN: 160 samples per mel frame (+32 tail)
    t = Tango.from_synthetic(unet_config=cfg, device=dev, precision=args.precision, scheduler=args.scheduler)
    if world > 1:
        # one-time NCCL broadcast of the (rank-0) weights over NVLink, as a sharded deployment would do at load
        usd = parallel.broadcast_state_dict({k: v.to(dev) for k, v in t.model.unet._sd.items()}, src=0)
        t.model.unet.load_state_dict(usd)
    embeds_h, mask_h = synthetic_inputs(B, args.tokens, cfg["cross_attention_dim"], rank)
    embeds_pin, mask_pin = embeds_h.pin_memory(), mask_h.pin_memory()
    embeds_d, mask_d = embeds_h.to(dev), mask_h.to(dev)
    prompts = [f"synthetic prompt {rank}-{i}" for i in range(B)]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)

    decode_ms = []
    last = {}   # the latest pass's outputs: persistent device buffers, overwritten by the next pass

    def one_pass_device():
        lat = t.model.inference(prompts, t.scheduler, args.denoise_steps, args.guidance, prompt_embeds=embeds_d,
                                boolean_prompt_mask=mask_d, generator=gen, latent_shape=latent_shape)
        B_, Cl, H, W = lat.shape
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        rows = lat.permute(0, 2, 3, 1).reshape(B_ * H * W, Cl).contiguous()
        out = t.vae.decode_rows_to_waveform(rows, B_, H, W)
        d1.record()
        decode_ms.append((d0, d1))
        last.update(latents=lat, waveform=out[0], waveform_int16=out[1])
        return out

    def one_pass_e2e():
        return t.generate_for_batch(prompts, steps=args.denoise_steps, guidance=args.guidance, batch_size=B,
                                    prompt_embeds=embeds_pin, boolean_prompt_mask=mask_pin, generator=gen,
                                    latent_shape=latent_shape)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- warm-up
    for _ in range(max(args.warmup, 1)):
        one_pass_device()
    barrier()
    # ---------------- timed: device-resident
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    n0 = L.launch_count()
    graph_launches = 0
    unet_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        one_pass_device()
        graph_launches += t.model.launches_per_forward * args.denoise_steps
        unet_ms.append(t.model.last_step_ms)
    ev1.record()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:   # before the legs below reuse the buffers
        dump_outputs(args.dump_outputs, last)
    launches = (L.launch_count() - n0) + graph_launches
    dec_ms = float(np.mean([a.elapsed_time(b) for a, b in decode_ms[-args.steps:]]))
    dev_ms = parallel.max_over_ranks(dev_ms, dev)
    value = world * B * audio_s * args.steps / (dev_ms / 1e3)

    # ---------------- timed: end to end through the public API with host buffers
    one_pass_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        waves = one_pass_e2e()
    barrier()
    e2e_s = parallel.max_over_ranks(time.perf_counter() - t0, dev)
    e2e_value = world * B * audio_s * args.steps / e2e_s
    h2d = embeds_pin.numel() * 4 + mask_pin.numel()
    d2h = sum(int(w.nbytes) for w in waves)

    # ---------------- BASELINE.json configs[3] / configs[4] at 8 GPUs (every rank takes part; rank 0 reports)
    extra = None
    if world == 8 and not args.no_extra_configs and args.unet == "base" and args.latent_h == 256:
        extra = extra_configs(args, dev, rank, world, barrier, t)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel: one instrumented (eager, CUDA-event-per-launch) UNet forward
    pk = peaks()
    m = t.model
    m.use_cuda_graph = False
    m.inference(prompts, t.scheduler, 1, args.guidance, prompt_embeds=embeds_d, boolean_prompt_mask=mask_d, generator=gen,
                latent_shape=latent_shape)
    torch.cuda.synchronize()
    # Park the GPU behind a ~0.25 s spin kernel so that the (slow, Python-driven) eager launches queue up ahead of the
    # GPU: the per-launch CUDA events then bracket pure kernel execution, not host launch latency.
    torch.cuda._sleep(int(0.25 * 1.9e9))
    L.PROF.start()
    m.inference(prompts, t.scheduler, 2, args.guidance, prompt_embeds=embeds_d, boolean_prompt_mask=mask_d, generator=gen,
                latent_shape=latent_shape)
    prof = L.PROF.stop()
    m.use_cuda_graph = True
    # gemm_tc_kernel families are labelled with the instantiation that ran (N tile, launch mode: lib.conv_gemm asks
    # tng_gemm_plan). The roofline block describes the DOMINANT one (largest share of the step); the whole family and
    # every other kernel follow in `kernel_families`.
    gfams = {k: v for k, v in prof.items() if k.startswith("gemm_tc")}
    gall = {"launches": sum(v["launches"] for v in gfams.values()), "ms": sum(v["ms"] for v in gfams.values()) or 1.0,
            "flops": sum(v["flops"] for v in gfams.values())}
    dom_name, gm = max(gfams.items(), key=lambda kv: kv[1]["ms"]) if gfams else ("gemm_tc", {"launches": 1, "ms": 1.0, "flops": 0.0})
    at = prof.get("attention_tc", {"launches": 1, "ms": 1.0, "flops": 0.0})
    achieved = gm["flops"] / (gm["ms"] / 1e3) / 1e12
    traffic = None      # dram bytes per launch of the dominant kernel: only ncu can measure it (profiles/, per round)
    for tp in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        tp = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            break
    roof = {"bound": "tensor", "kernel": f"{dom_name.replace('gemm_tc', 'gemm_tc_kernel')} (tcgen05 implicit-GEMM conv/linear; the "
                                         "instantiation with the largest share of the UNet step)",
            "achieved": achieved, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": achieved / pk["bf16_tflops_sustained"], "traffic": traffic,
            "peak_source": pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)",
            "launches_profiled": gm["launches"], "avg_launch_ms": gm["ms"] / max(1, gm["launches"]),
            "algorithmic_gflop_per_launch": gm["flops"] / max(1, gm["launches"]) / 1e9,
            "gemm_tc_all_instantiations": {"achieved": gall["flops"] / (gall["ms"] / 1e3) / 1e12,
                                           "frac": gall["flops"] / (gall["ms"] / 1e3) / 1e12 / pk["bf16_tflops_sustained"],
                                           "launches": gall["launches"], "ms_per_step": gall["ms"] / 2},
            "attention_tc": {"achieved": at["flops"] / (at["ms"] / 1e3) / 1e12, "launches": at["launches"],
                             "avg_launch_ms": at["ms"] / max(1, at["launches"])}}
    if args.latent_h == 256:
        f_unet, f_vae, f_voc = (F_UNET if args.unet == "base" else 806.453e9), F_VAE, F_VOC
    else:  # SURVEY.md §8d figures for the 30 s extension (768 x 16); other lengths are not tabulated
        f_unet, f_vae, f_voc = (3137.856e9 if args.unet == "base" else 3141.13e9), 2217.564e9, 3080.714e9
    f_total = B * (2 * args.denoise_steps * f_unet + f_vae + f_voc)
    whole = f_total * args.steps / (dev_ms / 1e3) / 1e12
    roof["whole_path_tflops"] = whole
    roof["whole_path_frac"] = whole / pk["bf16_tflops_sustained"]
    # every kernel family of the instrumented forwards (2 denoising steps): share of the step, achieved rate against the
    # roofline that bounds it (tensor families: algorithmic TFLOP/s; HBM families: algorithmic GB/s)
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    fam = {}
    for name, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        e = {"launches_per_step": v["launches"] / 2, "ms_per_step": v["ms"] / 2, "share": v["ms"] / tot_ms}
        if v["flops"] > 0:
            e["tflops"] = v["flops"] / (v["ms"] / 1e3) / 1e12
            e["frac_of_bf16_sustained"] = e["tflops"] / pk["bf16_tflops_sustained"]
        elif v["bytes"] > 0:
            e["gbs"] = v["bytes"] / (v["ms"] / 1e3) / 1e9
            e["frac_of_hbm"] = e["gbs"] / pk["hbm_gbs"]
        fam[name] = e
    roof["kernel_families"] = fam

    # ---------------- the mode that meets the north star's 1e-3 (precision="split"): its throughput on the same config,
    # and how far the timed bf16 mode drifts from it over the full 200-step chain on identical noise
    parity = None
    if world == 1 and not args.no_parity_mode and args.precision == "bf16":
        parity = parity_mode_leg(args, t, cfg, dev, prompts, embeds_d, mask_d, latent_shape, audio_s)

    # ---------------- text-conditioning front-end (SURVEY.md §8(f).1): reported beside the metric, not inside it
    # (BASELINE.json's metric excludes text encoding). FLAN-T5 encoder of the UNet's width, seeded random weights,
    # `batch` prompts x `tokens` tokens (the "" prompt is cached by the pipeline and not re-encoded).
    text = None
    if world == 1 and not args.no_text_encoder:          # like the CPU baseline: reported at N = 1 only
        text = text_encoder_leg(args, dev)

    # ---------------- CPU baseline (oracle port) on a bounded sample, N = 1 only
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args)

    line = {"metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "bf16x3 (split)",
            "data": "synthetic (seeded random weights of the Tango base architecture, random 64-token conditioning)",
            "config": workload_config(args, world), "unet_step_ms": float(np.mean(unet_ms)),
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
            "decode_ms": {"value": dec_ms, "what": f"VAE decoder + HiFi-GAN for {B} samples (one CUDA-graph replay), inside the timed pass"}}
    if parity is not None:
        line["parity_mode"] = parity
    if extra is not None:
        line["configs"] = extra
    if text is not None:
        line["text_encoder"] = text
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def parity_mode_leg(args, t_bf16, cfg, dev, prompts, embeds_d, mask_d, latent_shape, audio_s):
    from tango_b200.pipeline import Tango
    ts = Tango.from_synthetic(unet_config=cfg, device=dev, precision="split", scheduler=args.scheduler)

    def run(t, steps, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        lat = t.model.inference(prompts, t.scheduler, steps, args.guidance, prompt_embeds=embeds_d,
                                boolean_prompt_mask=mask_d, generator=g, latent_shape=latent_shape)
        B_, Cl, H, W = lat.shape
        rows = lat.permute(0, 2, 3, 1).reshape(B_ * H * W, Cl).contiguous()
        mel = t.vae.decode_rows(rows, B_, H, W).clone()
        wf, wi = t.vae.decode_rows_to_waveform(rows, B_, H, W)
        return lat.clone(), mel, wf.clone()

    run(ts, 3, 1)                                          # capture + warm-up at the same shapes
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    lat_s, mel_s, wav_s = run(ts, args.denoise_steps, 4321)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    lat_b, mel_b, wav_b = run(t_bf16, args.denoise_steps, 4321)
    torch.cuda.synchronize()

    def rel(a, b):
        return float((a.double() - b.double()).norm() / b.double().norm())

    # short chain for scale: the same comparison after 10 steps
    lat_s10, _, _ = run(ts, 10, 99)
    lat_b10, _, _ = run(t_bf16, 10, 99)
    out = {"precision": "split (bf16 hi/lo 3-term products on the tensor cores; GPU parity tests hold it to <= 1e-3 of the "
                        "fp32 reference: tests/test_config1_gpu.py)",
           "value": args.batch * audio_s / (ms / 1e3), "unit": "audio-s/s", "passes_timed": 1, "ms_per_pass": ms,
           "unet_step_ms": ts.model.last_step_ms,
           "bf16_vs_split": {"what": f"relative L2 distance of the timed bf16 mode from the split mode, same seed / noise, "
                                     f"{args.scheduler.upper()} chain",
                             "latents_after_10_steps": rel(lat_b10, lat_s10),
                             f"latents_after_{args.denoise_steps}_steps": rel(lat_b, lat_s),
                             "mel": rel(mel_b, mel_s), "waveform": rel(wav_b, wav_s)}}
    del ts
    torch.cuda.empty_cache()
    return out


def extra_configs(args, dev, rank, world, barrier, t_base):
    """BASELINE.json configs[3] (XL UNet, batch 32, 100 steps, 4 prompts per GPU) and configs[4] (base UNet, batch 64,
    200 steps, 30 s clips = 768 x 16 latents, 8 prompts per GPU) on the 8 GPUs: 2 timed passes each after one warm-up,
    device-timed, max over ranks, whole-job audio-s/s."""
    from tango_b200 import parallel, synth
    from tango_b200.pipeline import Tango
    out = {}
    specs = [("c4", "xl", 32, 100, 256), ("c5", "base", 64, 200, 768)]
    for name, unet, gbatch, steps, lh in specs:
        B = gbatch // world
        cfg = synth.BASE_UNET_CONFIG if unet == "base" else synth.XL_UNET_CONFIG
        t = t_base if unet == "base" else Tango.from_synthetic(unet_config=cfg, device=dev, precision=args.precision,
                                                               scheduler=args.scheduler)
        emb, msk = synthetic_inputs(B, args.tokens, cfg["cross_attention_dim"], 100 + rank)
        emb, msk = emb.to(dev), msk.to(dev)
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        prompts = [f"{name} prompt {rank}-{i}" for i in range(B)]
        audio_s = (4 * lh * 160 + 32) / 16000.0

        def one():
            lat = t.model.inference(prompts, t.scheduler, steps, args.guidance, prompt_embeds=emb, boolean_prompt_mask=msk,
                                    generator=gen, latent_shape=(lh, 16))
            B_, Cl, H, W = lat.shape
            rows = lat.permute(0, 2, 3, 1).reshape(B_ * H * W, Cl).contiguous()
            return t.vae.decode_rows_to_waveform(rows, B_, H, W)

        one()
        barrier()
        passes = 2
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(passes):
            one()
        e1.record()
        barrier()
        ms = parallel.max_over_ranks(e0.elapsed_time(e1), dev)
        out[name] = {"workload": f"Tango {unet} UNet, batch {gbatch} sharded {B}/GPU over {world} GPUs, {steps} "
                                 f"{args.scheduler.upper()} steps, CFG {args.guidance}, {audio_s:.2f} s clips, {args.precision}",
                     "value": gbatch * audio_s * passes / (ms / 1e3), "unit": "audio-s/s", "passes_timed": passes,
                     "ms_per_pass": ms / passes, "unet_step_ms": t.model.last_step_ms}
        if unet != "base":
            del t
            torch.cuda.empty_cache()
    return out


def text_encoder_leg(args, dev):
    from tango_b200 import synth
    from tango_b200.t5 import T5EncoderModel
    cfg = synth.FLAN_T5_LARGE_CONFIG if args.unet == "base" else synth.FLAN_T5_XL_CONFIG
    m = T5EncoderModel.from_config(cfg, precision=args.precision).to(dev)
    m.load_state_dict(synth.synth_state_dict(synth.t5_encoder_param_shapes(cfg), 0))
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(2, cfg["vocab_size"], (args.batch, args.tokens), generator=g).to(dev)
    mask = torch.ones(args.batch, args.tokens, dtype=torch.long, device=dev)
    for _ in range(2):
        m(ids, mask)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        m(ids, mask)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    rows, d, ff, inner = args.batch * args.tokens, cfg["d_model"], cfg["d_ff"], cfg["num_heads"] * cfg["d_kv"]
    flops = cfg["num_layers"] * (2 * rows * (4 * d * inner + 3 * d * ff) + 4 * args.batch * cfg["num_heads"] * args.tokens ** 2 * 64)
    del m
    torch.cuda.empty_cache()
    return {"model": ("flan-t5-large" if args.unet == "base" else "flan-t5-xl") + " encoder, seeded random weights",
            "prompts": args.batch, "tokens": args.tokens, "ms": ms, "tflops": flops / (ms / 1e3) / 1e12,
            "note": "one CUDA-graph replay per call; outside the timed metric"}


def cpu_baseline(args):
    """In-line CPU leg (N = 1): ONE measured denoising step at the benchmark batch + the decode of 2 of its samples
    (~30-60 s of CPU work on the box's physical cores) — same procedure and thread rule as --impl reference."""
    ref = CpuReference(args)
    t_step = ref.step_seconds(0)
    t_dec = ref.decode_seconds(2)
    audio_s = (4 * args.latent_h * 160 + 32) / 16000.0
    v = args.batch * audio_s / (args.denoise_steps * t_step + t_dec)
    return {"value": v, "unit": "audio-s/s", "cores": ref.cores, "kind": "port", "sample": ref.describe(t_step, 1, t_dec, 2)}


DUMP_LIMIT = 64 * 10**6   # bytes over all files written by --dump-outputs, .npy headers included


def dump_outputs(path, tensors):
    """Each tensor as path/<name>.npy in float32 (the int16 waveform converts exactly). The default workload writes
    ~11.5 MB; beyond DUMP_LIMIT every array is replaced by the same seeded random sample of its flattened elements, in
    proportion to its size, so that runs with the same arguments still compare element for element."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_LIMIT - 1024 * len(arrays)
    for name, a in arrays.items():
        if total > budget:
            k = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)
    print(f"bench.py: wrote {', '.join(sorted(arrays))} to {path}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="prompts per GPU")
    ap.add_argument("--denoise-steps", type=int, default=200)
    ap.add_argument("--guidance", type=float, default=3.0)
    ap.add_argument("--tokens", type=int, default=64)
    ap.add_argument("--scheduler", default="ddim", choices=["ddim", "ddpm"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "split"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-text-encoder", action="store_true", help="skip the FLAN-T5 front-end timing leg")
    ap.add_argument("--latent-h", type=int, default=256, help="latent time frames: 256 = 10.24 s (reference), 768 = 30.7 s")
    ap.add_argument("--unet", default="base", choices=["base", "xl"])
    ap.add_argument("--reference-budget-s", type=float, default=150.0,
                    help="--impl reference: stop timing further steps once this much wall time has been used")
    ap.add_argument("--no-parity-mode", action="store_true", help="skip the split-precision (1e-3 mode) leg")
    ap.add_argument("--no-extra-configs", action="store_true", help="at --gpus 8: skip the c4 / c5 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    knobs = sorted(k for k in os.environ if k.startswith("TNG_"))
    if knobs:
        raise SystemExit(f"bench.py: refusing to run with experiment knobs set in the environment: {knobs}")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
