"""Batch text-to-audio generation CLI — the caller side of the hot path (SURVEY.md section 8(f).3).

Mirrors /root/reference/inference_hf.py:30-119 (`--checkpoint --test_file --text_key --device --num_steps --guidance
--batch_size`, one JSON object per line in the prompt manifest, `outputs/<id>_steps_<n>_guidance_<g>/output_<j>.wav`
at 16 kHz PCM-16, one JSON line appended to `outputs/tango_checkpoint_summary.jsonl`), so the wav directory can be
scored by the reference's `audioldm_eval` unchanged. Differences, all additive:

  * `--checkpoint` is a local snapshot directory (no hub access) or `synthetic[:tiny|base|xl]` for seeded random weights;
  * under `torchrun` (one process per GPU) the prompts are split contiguously over the ranks, every rank writes the
    wavs of its own slice under their global indices, rank 0 writes the summary (no data-path collective);
  * objective metrics (FD / FAD / KL / IS through `audioldm_eval`, inference_hf.py:111) are out of scope: the summary
    carries generation facts and throughput instead; `--test_references` is accepted and recorded only.

    python -m tango_b200.cli --checkpoint /data/tango --test_file data/test_audiocaps_subset.json --num_steps 200
    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 -m tango_b200.cli --checkpoint /data/tango ...
"""
from __future__ import annotations

import argparse
import json
import os
import time
import wave
from typing import List, Optional, Sequence

import numpy as np


def parse_args(argv: Optional[Sequence[str]] = None) -> argparse.Namespace:
    p = argparse.ArgumentParser(description="Inference for text to audio generation task.")
    p.add_argument("--checkpoint", type=str, default="declare-lab/tango",
                   help="Local Tango snapshot directory, or synthetic[:tiny|base|xl]")
    p.add_argument("--test_file", type=str, default="data/test_audiocaps_subset.json",
                   help="json-lines file containing the test prompts for generation.")
    p.add_argument("--text_key", type=str, default="captions", help="Key containing the text in the json file.")
    p.add_argument("--device", type=str, default="cuda:0", help="Device to use for inference (single process).")
    p.add_argument("--test_references", type=str, default="data/audiocaps_test_references/subset",
                   help="Folder containing the test reference wav files (recorded in the summary only).")
    p.add_argument("--num_steps", type=int, default=200, help="How many denoising steps for generation.")
    p.add_argument("--guidance", type=float, default=3, help="Guidance scale for classifier free guidance.")
    p.add_argument("--batch_size", type=int, default=8, help="Batch size for generation.")
    # additive options
    p.add_argument("--output_root", type=str, default="outputs")
    p.add_argument("--exp_id", type=str, default=None, help="Run id (default: unix time; pass one under torchrun)")
    p.add_argument("--precision", default="bf16", choices=["bf16", "split"])
    p.add_argument("--scheduler", default="ddpm", choices=["ddpm", "ddim", "dpmsolver++"],
                   help="inference_hf.py uses DDPM; dpmsolver++ = DPM-Solver++ 2M, meant for 10-25 --num_steps")
    p.add_argument("--latent_h", type=int, default=256, help="latent frames: 256 = 10.24 s (reference)")
    p.add_argument("--seed", type=int, default=None, help="torch.manual_seed for reproducible noise")
    return p.parse_args(argv)


def read_prompts(path: str, text_key: str, prefix: str = "") -> List[str]:
    """inference_hf.py:86-87: one JSON object per line, `text_key` holds the caption."""
    out = []
    with open(path) as f:
        for line in f:
            if line.strip():
                out.append(prefix + json.loads(line)[text_key])
    return out


def write_wav(path: str, samples: np.ndarray, samplerate: int = 16000) -> None:
    """`sf.write(path, int16_array, samplerate=16000)` of inference_hf.py:107: mono PCM-16 RIFF."""
    a = np.asarray(samples)
    if a.dtype != np.int16:
        raise TypeError("write_wav expects the int16 waveform produced by the pipeline")
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(samplerate)
        w.writeframes(a.astype("<i2").tobytes())


def output_dir_for(root: str, exp_id: str, num_steps: int, guidance: float) -> str:
    return os.path.join(root, "{}_steps_{}_guidance_{}".format(exp_id, num_steps, guidance))


def build_tango(checkpoint: str, device: str, precision: str, scheduler: str):
    from . import synth
    from .pipeline import Tango
    if checkpoint.startswith("synthetic"):
        kind = checkpoint.split(":", 1)[1] if ":" in checkpoint else "base"
        ucfg = {"tiny": synth.TINY_UNET_CONFIG, "base": synth.BASE_UNET_CONFIG, "xl": synth.XL_UNET_CONFIG}[kind]
        return Tango.from_synthetic(ucfg, device=device, precision=precision, scheduler=scheduler)
    t = Tango(checkpoint, device, precision=precision)
    if scheduler == "ddim":
        from .schedulers import DDIMScheduler
        t.scheduler = DDIMScheduler.from_pretrained(t.scheduler_name, subfolder="scheduler")   # same scheduler_config.json
    elif scheduler == "dpmsolver++":
        from .schedulers import DPMSolverMultistepScheduler
        t.scheduler = DPMSolverMultistepScheduler.from_config(t.scheduler.config)   # same betas / prediction type
    return t


def main(argv: Optional[Sequence[str]] = None) -> dict:
    import torch
    from . import parallel
    args = parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    device = args.device
    if world > 1:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        device = f"cuda:{local}"
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group("nccl")
        if args.exp_id is None:       # every rank must agree on the directory name
            t = torch.tensor([int(time.time())], device=device)
            dist.broadcast(t, 0)
            args.exp_id = str(int(t.item()))
    if args.seed is not None:
        # the SAME seed on every rank: each rank draws the full-batch noise and keeps its rows, so an N-GPU run produces
        # the waveforms of the one-GPU run (SURVEY.md section 8e, AudioDiffusion.randn_rows)
        torch.manual_seed(args.seed)

    prompts = read_prompts(args.test_file, args.text_key)
    exp_id = args.exp_id or str(int(time.time()))
    out_dir = output_dir_for(args.output_root, exp_id, args.num_steps, args.guidance)
    os.makedirs(out_dir, exist_ok=True)

    tango = build_tango(args.checkpoint, device, args.precision, args.scheduler)
    kw = {} if args.latent_h == 256 else {"latent_shape": (args.latent_h, 16)}
    torch.cuda.synchronize()
    t0 = time.time()
    # every chunk of batch_size prompts is split over the ranks; all ranks end up with all waveforms
    waves = tango.generate_for_batch(prompts, steps=args.num_steps, guidance=args.guidance,
                                     batch_size=args.batch_size, shard=world > 1, **kw)
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    for j, wav in enumerate(waves):
        if j % world == rank:                     # the file writes are spread over the ranks
            write_wav(os.path.join(out_dir, "output_{}.wav".format(j)), wav)
    if world > 1:
        gen_s = parallel.max_over_ranks(gen_s, device)
    audio_s = sum(len(w) for w in waves) / 16000.0

    result = {"Steps": args.num_steps, "Guidance Scale": args.guidance, "Test Instances": len(prompts),
              "scheduler_config": dict(tango.scheduler.config), "args": dict(vars(args)), "output_dir": out_dir,
              "n_gpus": world, "generation_seconds": gen_s, "audio_seconds": audio_s,
              "audio_seconds_per_second": audio_s / max(gen_s, 1e-9),
              "text_encoder": "synthetic" if getattr(tango.model.text_encoder, "synthetic", False) else "t5",
              "tokenizer": "synthetic" if getattr(getattr(tango.model, "tokenizer", None), "synthetic", False) else
                           ("n/a" if getattr(tango.model, "tokenizer", None) is None else "t5"),
              "metrics": "not computed here: score output_dir with audioldm_eval as inference_hf.py:111 does"}
    if rank == 0:
        with open(os.path.join(args.output_root, "tango_checkpoint_summary.jsonl"), "a") as f:
            f.write(json.dumps(result) + "\n\n")
        print(json.dumps({k: result[k] for k in ("output_dir", "Test Instances", "audio_seconds_per_second")}))
    return result


if __name__ == "__main__":
    main()
