"""AudioDiffusion.inference and the Tango façade on the B200 kernels.

Mirrors /root/reference/models.py:210-305 (`AudioDiffusion.inference`, `prepare_latents`,
`encode_text_classifier_free`) and /root/reference/tango.py:9-64 (`Tango.generate`, `generate_for_batch`, `chunks`):
same names, argument meaning, defaults and return types. What changes underneath:

  * the whole UNet forward is one CUDA-graph replay of hand-written sm_100a kernels (tango_b200/unet.py);
  * cross-attention K/V and the time-embedding projections are computed once per call, not once per step;
  * CFG combine + scheduler update + re-packing of the next UNet input are ONE kernel (tng_sched_step, or
    tng_sched_multistep for DPMSolverMultistepScheduler) fed from a per-step coefficient table and launched by the
    scheduler's `fused_step`, so there is no host sync inside the loop (the reference has two per step);
  * a prompt batch can be sharded over the GPUs of one box (tango_b200/parallel.py) — samples are independent.

Text encoding (SURVEY.md §8(f).1): the FLAN-T5 encoder runs on the same kernels (tango_b200/t5.py) whenever its
weights are present (`text_encoder.*` of pytorch_model_main.bin, or a local snapshot directory); the unconditional
("") embedding is computed once per padded length and reused. Tokenisation stays on the host (AutoTokenizer from a
local snapshot; a flagged stand-in tokenizer when SentencePiece data is not reachable). Without any encoder weights a
flagged synthetic encoder supplies conditioning of the right shape; tests and the benchmark may also inject
`prompt_embeds` directly.
"""
from __future__ import annotations

import json
import os
import warnings
import zlib
from collections import OrderedDict
from types import SimpleNamespace
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import lib as L
from . import parallel
from . import synth
from .schedulers import DDIMScheduler, DDPMScheduler, DPMSolverMultistepScheduler
from .stft import TacotronSTFT
from .t5 import T5EncoderModel
from .unet import UNet2DConditionModel
from .vae import AutoencoderKL

LATENT_HW = (256, 16)  # models.py:259-260 (10.24 s); `latent_shape` may override (30 s clips: (768, 16))


class SyntheticTextEncoder:
    """Deterministic stand-in for FLAN-T5 when no checkpoint is reachable: embeddings are a seeded function of the
    prompt string (dense Gaussian, like T5 states), padded to the longest prompt of the batch with a proper mask."""

    synthetic = True

    def __init__(self, dim: int, tokens: int = 64):
        self.dim, self.tokens = dim, tokens

    def encode(self, prompts: Sequence[str], fixed_len: Optional[int] = None):
        lens = [min(self.tokens, max(1, len(p.split()) + 1)) if p else 1 for p in prompts]
        Lmax = fixed_len or (max(lens) if any(prompts) else 1)
        emb = torch.zeros(len(prompts), Lmax, self.dim)
        mask = torch.zeros(len(prompts), Lmax, dtype=torch.long)
        for i, p in enumerate(prompts):
            g = torch.Generator().manual_seed(zlib.crc32(p.encode()) & 0x7FFFFFFF)
            n = min(lens[i], Lmax)
            emb[i] = torch.randn(Lmax, self.dim, generator=g)
            mask[i, :n] = 1
        return emb, mask


class FallbackTokenizer:
    """Stand-in for the FLAN-T5 SentencePiece tokenizer when its `spiece.model` is not reachable (offline box): words
    are hashed into the vocabulary, EOS (id 1) is appended, pad id is 0 — the call signature and the padding /
    truncation behaviour the reference relies on (models.py:131-133, 268-286) are kept, the ids themselves are NOT
    T5's. Flagged `.synthetic`; with a real snapshot directory `AutoTokenizer` is used instead."""

    synthetic = True
    model_max_length = 512

    def __init__(self, vocab_size: int):
        self.vocab_size = vocab_size

    def __call__(self, prompts, max_length=None, padding=True, truncation=True, return_tensors="pt"):
        max_length = max_length or self.model_max_length
        rows = []
        for p in prompts:
            ids = [2 + zlib.crc32(w.encode()) % (self.vocab_size - 2) for w in p.split()] + [1]
            if truncation and len(ids) > max_length:
                ids = ids[:max_length - 1] + [1]
            rows.append(ids)
        width = max_length if padding == "max_length" else max(len(r) for r in rows)
        input_ids = torch.zeros(len(rows), width, dtype=torch.long)
        mask = torch.zeros(len(rows), width, dtype=torch.long)
        for i, r in enumerate(rows):
            input_ids[i, :len(r)] = torch.tensor(r)
            mask[i, :len(r)] = 1
        return SimpleNamespace(input_ids=input_ids, attention_mask=mask)


def t5_config_from_state_dict(te: dict) -> dict:
    """Encoder hyper-parameters recovered from `text_encoder.*` tensor shapes (pytorch_model_main.bin carries no config)."""
    emb = te["shared.weight"] if "shared.weight" in te else te["encoder.embed_tokens.weight"]
    layers = 1 + max(int(k.split(".")[2]) for k in te if k.startswith("encoder.block."))
    inner = te["encoder.block.0.layer.0.SelfAttention.q.weight"].shape[0]
    buckets, heads = te["encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"].shape
    return {"vocab_size": emb.shape[0], "d_model": emb.shape[1], "d_kv": inner // heads, "num_heads": heads,
            "d_ff": te["encoder.block.0.layer.1.DenseReluDense.wi_0.weight"].shape[0], "num_layers": layers,
            "relative_attention_num_buckets": buckets, "relative_attention_max_distance": 128,
            "layer_norm_epsilon": 1e-6, "feed_forward_proj": "gated-gelu"}


class AudioDiffusion:
    """Inference half of /root/reference/models.py:AudioDiffusion (the training half, :105-208, is out of scope)."""

    def __init__(self, text_encoder_name=None, scheduler_name=None, unet_model_name=None,
                 unet_model_config_path=None, snr_gamma=None, freeze_text_encoder=True, uncondition=False,
                 unet_config: Optional[dict] = None, precision: str = "bf16", use_cuda_graph: bool = True,
                 allow_synthetic_tokenizer: bool = False):
        assert unet_model_config_path is not None or unet_config is not None or unet_model_name is not None, \
            "Either UNet pretrain model name or a config file path is required"
        if unet_model_name is not None and unet_config is None and unet_model_config_path is None:
            raise NotImplementedError("set_from='pre-trained' (Stable-Diffusion UNet + group_in/out) is an ablation of the"
                                      " reference (models.py:88-93) and not on the accelerated path")
        self.text_encoder_name, self.scheduler_name = text_encoder_name, scheduler_name
        self.unet_model_config_path, self.snr_gamma = unet_model_config_path, snr_gamma
        self.freeze_text_encoder, self.uncondition = freeze_text_encoder, uncondition
        cfg = unet_config if unet_config is not None else UNet2DConditionModel.load_config(unet_model_config_path)
        self.unet = UNet2DConditionModel.from_config(cfg, precision=precision)
        self.set_from = "random"
        self.precision = precision
        self.use_cuda_graph = use_cuda_graph
        self.noise_scheduler = DDPMScheduler.from_pretrained(scheduler_name, subfolder="scheduler")
        self.inference_scheduler = DDPMScheduler.from_pretrained(scheduler_name, subfolder="scheduler")
        self.device = torch.device("cpu")
        self.tokenizer = None
        self.text_encoder = None
        self.allow_synthetic_tokenizer = allow_synthetic_tokenizer   # tests / synthetic weights only (see below)
        self._uncond_cache = {}
        self._state = OrderedDict()   # captured CUDA graphs + their persistent I/O buffers, LRU-bounded
        self._temb_cache = {}
        self.last_step_ms: Optional[float] = None
        self.last_kernel_launches = 0
        self.launches_per_forward = 0

    # ------------------------------------------------------------------------------------------ module plumbing
    MAX_GRAPHS = 8      # distinct (batch, clip length, padded text length, ...) shapes kept captured
    LK_BUCKET = 32      # masked text lengths are padded up to a multiple of this (one graph per bucket, not per length)

    def _invalidate(self):
        """Captured graphs hold raw pointers into the UNet's packed weights and scratch buffers: drop them whenever
        those are rebuilt (new weights, new device)."""
        self._state.clear()
        self._temb_cache = {}

    def to(self, device):
        if torch.device(device) != self.device:
            self._invalidate()
        self.device = torch.device(device)
        self.unet.to(self.device)
        if self.text_encoder is not None and hasattr(self.text_encoder, "to"):
            self.text_encoder.to(self.device)
        return self

    def eval(self):
        return self

    def load_state_dict(self, sd, strict: bool = True):
        """pytorch_model_main.bin holds `unet.*` and `text_encoder.*` keys (tango.py:28, SURVEY.md §3.3)."""
        unet_sd = {k[len("unet."):]: v for k, v in sd.items() if k.startswith("unet.")}
        self.unet.load_state_dict(unet_sd, strict=strict)
        self._invalidate()
        te = {k[len("text_encoder."):]: v for k, v in sd.items() if k.startswith("text_encoder.")}
        if te:
            self.set_text_encoder_state_dict(te)
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    def set_text_encoder_state_dict(self, te: dict, config: Optional[dict] = None):
        """Build the FLAN-T5 encoder (tango_b200.t5.T5EncoderModel, on the kernels) from `text_encoder.*` weights."""
        self.text_encoder = T5EncoderModel.from_config(config or t5_config_from_state_dict(te),
                                                       precision=self.precision).to(self.device)
        self.text_encoder.load_state_dict(te, strict=False)
        self._uncond_cache = {}

    def _ensure_text_encoder(self):
        """Tokenizer: AutoTokenizer from a local snapshot of `text_encoder_name`, else the flagged FallbackTokenizer.
        Encoder: the one built from `text_encoder.*` weights (load_state_dict), else a local snapshot directory, else
        the flagged SyntheticTextEncoder (no weights reachable offline)."""
        name = self.text_encoder_name or ""
        if self.text_encoder is None and os.path.isdir(name) and os.path.exists(os.path.join(name, "config.json")):
            self.text_encoder = T5EncoderModel.from_pretrained(name, precision=self.precision).to(self.device)
        if self.text_encoder is None:
            self.text_encoder = SyntheticTextEncoder(self.unet.config["cross_attention_dim"])
        if self.tokenizer is None and not getattr(self.text_encoder, "synthetic", False):
            try:
                from transformers import AutoTokenizer
                self.tokenizer = AutoTokenizer.from_pretrained(name, local_files_only=True)
            except Exception as e:
                # A real FLAN-T5 encoder fed with hashed token ids produces meaningless conditioning: refuse unless the
                # caller opted in (tests and seeded random weights, where the ids carry no meaning anyway).
                if not self.allow_synthetic_tokenizer:
                    raise L.TangoB200Error(
                        f"the FLAN-T5 tokenizer of '{name}' is not available locally ({type(e).__name__}: {e}); pass a "
                        "snapshot directory that contains its SentencePiece files, or construct AudioDiffusion with "
                        "allow_synthetic_tokenizer=True (synthetic weights / tests only)") from e
                warnings.warn("tango_b200: using the hashed stand-in tokenizer (FallbackTokenizer): token ids are NOT "
                              "FLAN-T5's — only meaningful with synthetic weights", stacklevel=2)
                self.tokenizer = FallbackTokenizer(self.text_encoder.cfg["vocab_size"])

    # ------------------------------------------------------------------------------------------ text (boundary input)
    def encode_text(self, prompt: List[str]):
        """models.py:129-147."""
        self._ensure_text_encoder()
        if getattr(self.text_encoder, "synthetic", False):
            emb, mask = self.text_encoder.encode(prompt)
            return emb.to(self.device), (mask == 1).to(self.device)
        batch = self.tokenizer(prompt, max_length=self.tokenizer.model_max_length, padding=True, truncation=True,
                               return_tensors="pt")
        ids, am = batch.input_ids.to(self.device), batch.attention_mask.to(self.device)
        with torch.no_grad():
            hs = self.text_encoder(input_ids=ids, attention_mask=am)[0]
        return hs, (am == 1).to(self.device)

    def encode_text_classifier_free(self, prompt: List[str], num_samples_per_prompt: int):
        """models.py:266-305: returns ([uncond; cond] embeddings (2B, L, D), bool mask (2B, L))."""
        self._ensure_text_encoder()
        if getattr(self.text_encoder, "synthetic", False):
            emb, am = self.text_encoder.encode(prompt)
            nemb, nam = self.text_encoder.encode([""] * len(prompt), fixed_len=emb.shape[1])
        else:
            batch = self.tokenizer(prompt, max_length=self.tokenizer.model_max_length, padding=True, truncation=True,
                                   return_tensors="pt")
            ids, am = batch.input_ids.to(self.device), batch.attention_mask.to(self.device)
            with torch.no_grad():
                emb = self.text_encoder(input_ids=ids, attention_mask=am)[0]
            # the "" prompt encodes to the same tensor for every sample and call: run it once per padded length
            key = int(emb.shape[1])
            hit = self._uncond_cache.get(key)
            if hit is None:
                ub = self.tokenizer([""], max_length=key, padding="max_length", truncation=True, return_tensors="pt")
                uids, uam = ub.input_ids.to(self.device), ub.attention_mask.to(self.device)
                with torch.no_grad():
                    hit = (self.text_encoder(input_ids=uids, attention_mask=uam)[0], uam)
                self._uncond_cache[key] = hit
            nemb, nam = hit[0].expand(len(prompt), -1, -1), hit[1].expand(len(prompt), -1)
        emb = emb.repeat_interleave(num_samples_per_prompt, 0)
        am = am.repeat_interleave(num_samples_per_prompt, 0)
        nemb = nemb.repeat_interleave(num_samples_per_prompt, 0)
        nam = nam.repeat_interleave(num_samples_per_prompt, 0)
        pe = torch.cat([nemb, emb]).to(self.device)
        pm = torch.cat([nam, am]).to(self.device)
        return pe, (pm == 1)

    @staticmethod
    def randn_rows(shape, generator, device, dtype=torch.float32, rows=None) -> torch.Tensor:
        """The seed contract of diffusers' `randn_tensor` (D/utils/torch_utils.py:29-70) plus the sharding rule of
        SURVEY.md section 8e. `generator`: None (global torch RNG), one torch.Generator, or a LIST with one generator
        per sample — then every sample is drawn on its own as a (1, ...) tensor and the draws are concatenated
        (torch_utils.py:60-66), which makes a sample's noise independent of batch size, chunking and GPU count.
        `rows` = (lo, hi, total): this process holds samples [lo, hi) of a `total`-sample batch. With a single
        generator the FULL (total, ...) tensor is drawn and sliced, so that every rank (same seed) sees exactly the
        stream a one-GPU run would; with a per-sample list only the local generators [lo, hi) are consumed."""
        lo, hi, total = (0, shape[0], shape[0]) if rows is None else rows
        if hi - lo != shape[0]:
            raise ValueError(f"rows={rows} does not match a local batch of {shape[0]}")
        if isinstance(generator, (list, tuple)):
            if len(generator) == 1:
                generator = generator[0]
            elif len(generator) == total:
                generator = list(generator[lo:hi])
            elif len(generator) != shape[0]:
                raise ValueError(f"You have passed a list of generators of length {len(generator)}, but requested an "
                                 f"effective batch size of {total}. Make sure the batch size matches the length of "
                                 "the generators.")
        if isinstance(generator, (list, tuple)):
            one = (1,) + tuple(shape[1:])
            parts = [torch.randn(one, generator=g, device=g.device, dtype=dtype).to(device) for g in generator]
            return torch.cat(parts, dim=0)
        gdev = device if generator is None else generator.device
        full = torch.randn((total,) + tuple(shape[1:]), generator=generator, device=gdev, dtype=dtype).to(device)
        return full if (lo == 0 and hi == total) else full[lo:hi].contiguous()

    def advance_rng(self, total_batch, inference_scheduler, num_steps, generator=None, latent_shape=LATENT_HW):
        """Consume exactly the random numbers `inference` would for a `total_batch`-sample batch without running it:
        a rank whose shard of a chunk is empty calls this so that its (shared-seed) stream stays aligned with the
        one-GPU run for the chunks that follow. Per-sample generator lists need nothing."""
        if isinstance(generator, (list, tuple)) and len(generator) > 1:
            return
        if isinstance(generator, (list, tuple)):
            generator = generator[0]
        sch = inference_scheduler
        sch.set_timesteps(num_steps, device=self.device)
        gdev = self.device if generator is None else generator.device
        shape = (total_batch, self.unet.config["in_channels"], *latent_shape)
        torch.randn(shape, generator=generator, device=gdev, dtype=torch.float32)
        for i in range(len(sch.timesteps)):
            if sch._needs_noise(sch.timestep_at(i)):
                torch.randn(shape, generator=generator, device=gdev, dtype=torch.float32)

    def prepare_latents(self, batch_size, inference_scheduler, num_channels_latents, dtype, device, generator=None,
                        latent_shape=LATENT_HW, rows=None):
        """models.py:259-264."""
        shape = (batch_size, num_channels_latents, *latent_shape)
        latents = self.randn_rows(shape, generator, device, dtype, rows)
        return latents * inference_scheduler.init_noise_sigma

    # ------------------------------------------------------------------------------------------ the hot loop
    @torch.no_grad()
    def inference(self, prompt, inference_scheduler, num_steps=20, guidance_scale=3, num_samples_per_prompt=1,
                  disable_progress=True, *, prompt_embeds: Optional[torch.Tensor] = None,
                  boolean_prompt_mask: Optional[torch.Tensor] = None, latents: Optional[torch.Tensor] = None,
                  noises: Optional[Sequence[torch.Tensor]] = None, generator=None, latent_shape=LATENT_HW,
                  trace: Optional[list] = None, extra_streams=(), noise_rows=None) -> torch.Tensor:
        """models.py:210-257. Extra keyword-only arguments (all optional): inject conditioning (`prompt_embeds`
        [(2)B, L, D] + `boolean_prompt_mask`), initial `latents`, per-step `noises` (one (B,8,H,W) tensor per step,
        used where the reference draws randn) or a torch `generator` (or a list with one generator per sample, as
        diffusers' randn_tensor accepts); `noise_rows` = (lo, hi, total) when this process holds samples [lo, hi) of a
        `total`-sample batch sharded over GPUs (see randn_rows); `latent_shape` for clips other than 10 s;
        `extra_streams` = ((encoded beats [(2)B, L, D], mask), (encoded chords, mask)) turns the loop into Mustango's
        MusicAudioDiffusion.inference (mustango/models.py:540-600; needs a UNet config with the *Music blocks)."""
        device = self.device
        L.require_cuda_device(device)   # no CPU fallback
        cfg_on = guidance_scale > 1.0
        if prompt_embeds is None:
            if cfg_on:
                prompt_embeds, boolean_prompt_mask = self.encode_text_classifier_free(prompt, num_samples_per_prompt)
            else:
                prompt_embeds, boolean_prompt_mask = self.encode_text(prompt)
                prompt_embeds = prompt_embeds.repeat_interleave(num_samples_per_prompt, 0)
                boolean_prompt_mask = boolean_prompt_mask.repeat_interleave(num_samples_per_prompt, 0)
        Bu = prompt_embeds.shape[0]
        batch_size = Bu // 2 if cfg_on else Bu
        sch = inference_scheduler
        sch.set_timesteps(num_steps, device=device)
        timesteps = sch.timesteps
        Cl = self.unet.config["in_channels"]
        H, W = latent_shape
        if latents is None:
            latents = self.prepare_latents(batch_size, sch, Cl, torch.float32, device, generator, latent_shape,
                                           rows=noise_rows)
        else:
            latents = latents.to(device, torch.float32) * sch.init_noise_sigma
        sample = latents.contiguous().clone()

        unet = self.unet
        if boolean_prompt_mask is not None and prompt_embeds.shape[1] % self.LK_BUCKET:
            # pad the text length up to the bucket: masked keys get the reference's -10000 bias (exp underflows to
            # exactly 0 in fp32), so the result is unchanged while real traffic needs one graph per bucket, not per length
            pad = self.LK_BUCKET - prompt_embeds.shape[1] % self.LK_BUCKET
            prompt_embeds = torch.nn.functional.pad(prompt_embeds, (0, 0, 0, pad))
            if boolean_prompt_mask.dtype is torch.bool:
                boolean_prompt_mask = torch.nn.functional.pad(boolean_prompt_mask, (0, pad), value=False)
            else:   # any other dtype is already an additive bias (unet_2d_condition.py:573-578): padded keys get -10000
                boolean_prompt_mask = torch.nn.functional.pad(boolean_prompt_mask, (0, pad), value=-10000.0)
        unet.set_conditioning(prompt_embeds, boolean_prompt_mask, extra_streams=extra_streams)
        tkey = (unet.pack_generation, str(device)) + tuple(sch._t_list)   # packed weights are rebuilt on (re)load
        if self._temb_cache.get("key") != tkey:   # batch- and data-independent: reuse across calls with the same grid
            self._temb_cache = {"key": tkey, "table": unet.time_embedding_table(timesteps)}
        temb_table = self._temb_cache["table"]                      # [steps, temb_total]
        s = unet.s
        HW = H * W
        # cfg_on is part of the key: the captured forward bakes in cfg_shared (the CFG shared prefix); so are the device
        # and the generation of the packed weights the graph points into
        key = (Bu, H, W, prompt_embeds.shape[1], boolean_prompt_mask is not None, bool(cfg_on), str(device),
               unet.pack_generation) + tuple((f.shape[1], m is not None) for f, m in extra_streams)
        st = self._state.get(key)
        if st is not None:
            self._state.move_to_end(key)
        if st is None:
            while len(self._state) >= self.MAX_GRAPHS:
                self._state.popitem(last=False)
            st = SimpleNamespace(
                x_in=torch.zeros(Bu * HW, Cl * s, device=device, dtype=torch.bfloat16),
                model_out=torch.zeros(Bu * HW, unet.config["out_channels"], device=device, dtype=torch.float32),
                temb_cur=torch.zeros(Bu, temb_table.shape[1], device=device, dtype=torch.float32),
                ident=torch.tensor([0, 0, 0, 1, 0, 0, 0, 0, 0, 1], device=device, dtype=torch.float32),
                graph=None, per_forward=0)
            self._state[key] = st
        x_in, model_out, temb_cur = st.x_in, st.model_out, st.temb_cur
        so = Cl if unet.split else 0
        # pack the initial latents into the (CFG-duplicated) channels-last bf16 UNet input
        L.sched_step(None, cfg_on, float(guidance_scale), sample, None, st.ident, None, x_in, B=batch_size, Cc=Cl, HW=HW,
                     split_off=so)

        def run_unet():
            unet.forward_rows(x_in, Bu, H, W, temb_cur, temb_cur.shape[1], out=model_out, cfg_shared=cfg_on)

        graph = None
        per_forward = 0
        if self.use_cuda_graph:
            if st.graph is None:
                # the whole UNet forward (~400 launches) is captured once per shape; all its operands live in
                # persistent buffers, so later calls only refresh their contents and replay
                temb_cur.copy_(temb_table[0:1].expand_as(temb_cur))
                n0 = L.launch_count()
                run_unet()  # warm-up: allocates every scratch buffer, sets kernel attributes
                st.per_forward = L.launch_count() - n0
                torch.cuda.synchronize()
                st.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(st.graph):
                    run_unet()
            graph, per_forward = st.graph, st.per_forward
        self.launches_per_forward = per_forward
        n_eager0 = L.launch_count()

        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(len(timesteps)):
            temb_cur.copy_(temb_table[i:i + 1].expand_as(temb_cur))
            if graph is not None:
                graph.replay()
            else:
                run_unet()
            noise = None
            if sch._needs_noise(sch.timestep_at(i)):
                if noises is not None:
                    noise = noises[i].to(device, torch.float32).contiguous()
                else:
                    noise = self.randn_rows((batch_size, Cl, H, W), generator, device, torch.float32, noise_rows)
            sch.fused_step(i, model_out, cfg_on, float(guidance_scale), sample, noise, x_in, B=batch_size, Cc=Cl, HW=HW,
                           split_off=so)
            if trace is not None:
                trace.append(sample.clone())
        ev1.record()
        torch.cuda.synchronize()
        self.last_step_ms = ev0.elapsed_time(ev1) / max(1, len(timesteps))
        # kernels of libtango_b200.so executed by this call (graph replays re-run the captured launches)
        self.last_kernel_launches = (L.launch_count() - n_eager0) + (per_forward * len(timesteps) if graph is not None else 0)
        return sample


class Tango:
    """tango.py:9-64. `name` is a local directory with the reference's checkpoint layout (vae_config.json,
    stft_config.json, main_config.json, pytorch_model_{vae,stft,main}.bin); the hub download of the reference needs
    network access and is replaced by that local path. `Tango.from_synthetic()` builds a random-weight instance."""

    def __init__(self, name="declare-lab/tango", device="cuda:0", precision: str = "bf16", unet_config_path=None):
        path = name
        if not os.path.isdir(path):
            raise FileNotFoundError(
                f"'{name}' is not a local checkpoint directory. The reference downloads it from the Hugging Face hub "
                "(tango.py:12); offline, pass the directory of a downloaded snapshot or use Tango.from_synthetic().")
        vae_config = json.load(open(f"{path}/vae_config.json"))
        stft_config = json.load(open(f"{path}/stft_config.json"))
        main_config = json.load(open(f"{path}/main_config.json"))
        if unet_config_path is not None:
            main_config["unet_model_config_path"] = unet_config_path
        self._init_modules(vae_config, main_config, device, precision, stft_config=stft_config)
        self.vae.load_state_dict(torch.load(f"{path}/pytorch_model_vae.bin", map_location="cpu"))
        self.stft.load_state_dict(torch.load(f"{path}/pytorch_model_stft.bin", map_location="cpu"))
        self.model.load_state_dict(torch.load(f"{path}/pytorch_model_main.bin", map_location="cpu"))
        print("Successfully loaded checkpoint from:", name)

    def _init_modules(self, vae_config, main_config, device, precision, unet_config=None, stft_config=None,
                      allow_synthetic_tokenizer: bool = False):
        self.device = torch.device(device)
        self.vae = AutoencoderKL(**vae_config, precision=precision).to(device)
        # tango.py:19,23,27 — read by inference.py:81 / inference_hf.py:77 (tango.stft): the mel front-end on the kernels
        self.stft = TacotronSTFT(**(stft_config or synth.STFT_CONFIG)).to(device)
        mc = {k: v for k, v in main_config.items()}
        self.model = AudioDiffusion(**mc, unet_config=unet_config, precision=precision,
                                    allow_synthetic_tokenizer=allow_synthetic_tokenizer).to(device)
        self.vae.eval()
        self.stft.eval()
        self.model.eval()
        self.scheduler_name = main_config.get("scheduler_name")
        self.scheduler = DDPMScheduler.from_pretrained(self.scheduler_name, subfolder="scheduler")

    @classmethod
    def from_synthetic(cls, unet_config: Optional[dict] = None, device="cuda:0", precision: str = "bf16", seed: int = 0,
                       scheduler: str = "ddpm", t5_config: Optional[dict] = None):
        """Random-weight instance with the reference's architecture (no checkpoint is reachable offline). With
        `t5_config` (e.g. synth.FLAN_T5_LARGE_CONFIG) a random-weight FLAN-T5 encoder of that shape is attached too, so
        prompts run through tokenizer -> T5 kernels -> UNet instead of the synthetic conditioning stand-in."""
        self = cls.__new__(cls)
        ucfg = dict(unet_config or synth.BASE_UNET_CONFIG)
        self._init_modules(dict(synth.VAE_CONFIG), {"scheduler_name": "stabilityai/stable-diffusion-2-1",
                                                    "text_encoder_name": None}, device, precision, unet_config=ucfg,
                           allow_synthetic_tokenizer=True)
        self.model.unet.load_state_dict(synth.synth_state_dict(synth.unet_param_shapes(ucfg), seed))
        self.vae.load_state_dict(synth.synth_state_dict(synth.vae_decoder_param_shapes(), seed))
        if scheduler == "ddim":
            self.scheduler = DDIMScheduler.from_pretrained(None)
        elif scheduler == "dpmsolver++":   # DPM-Solver++ 2M (midpoint) with the SD-2.1 betas / v_prediction
            self.scheduler = DPMSolverMultistepScheduler.from_pretrained(None)
        if t5_config is not None:
            if t5_config["d_model"] != ucfg["cross_attention_dim"]:
                raise ValueError("t5_config['d_model'] must equal the UNet's cross_attention_dim")
            self.model.set_text_encoder_state_dict(
                synth.synth_state_dict(synth.t5_encoder_param_shapes(t5_config), seed), config=t5_config)
        return self

    def chunks(self, lst, n):
        """ Yield successive n-sized chunks from a list. """
        for i in range(0, len(lst), n):
            yield lst[i:i + n]

    def _decode(self, latents: torch.Tensor) -> np.ndarray:
        """decode_first_stage + decode_to_waveform without leaving channels-last rows (tango.py:47-48)."""
        B, Cl, H, W = latents.shape
        rows = latents.float().permute(0, 2, 3, 1).reshape(B * H * W, Cl).contiguous()
        _, wi = self.vae.decode_rows_to_waveform(rows, B, H, W, use_cuda_graph=self.model.use_cuda_graph)
        return wi.cpu().numpy()

    def generate(self, prompt, steps=100, guidance=3, samples=1, disable_progress=True, **kw):
        """ Genrate audio for a single prompt string. """
        with torch.no_grad():
            latents = self.model.inference([prompt], self.scheduler, steps, guidance, samples,
                                           disable_progress=disable_progress, **kw)
            wave = self._decode(latents)
        return wave[0]

    def generate_for_batch(self, prompts, steps=100, guidance=3, samples=1, batch_size=8, disable_progress=True,
                           shard: bool = False, **kw):
        """ Genrate audio for a list of prompt strings. With `shard=True` under torch.distributed every chunk of
        `batch_size` prompts is split contiguously over the ranks (SURVEY.md section 8e) and every rank returns all
        waveforms. The noise of a sharded run equals that of the one-GPU run on the same seed: each rank draws the
        chunk's full-batch tensors from its (identically seeded) generator and keeps its rows, or consumes only its own
        entries of a per-sample `generator` list (AudioDiffusion.randn_rows; diffusers torch_utils.py:29-70)."""
        prompts = list(prompts)
        world, r = (parallel.world_size(), parallel.rank()) if shard else (1, 0)
        gens = kw.pop("generator", None)
        per_sample = isinstance(gens, (list, tuple)) and len(gens) > 1
        if per_sample and len(gens) != len(prompts) * samples:
            raise ValueError(f"a per-sample generator list needs {len(prompts) * samples} entries, got {len(gens)}")
        outputs = []
        for k in range(0, len(prompts), batch_size):
            batch = prompts[k: k + batch_size]
            lo, hi = parallel.shard_range(len(batch), r, world)
            g = list(gens[k * samples:(k + len(batch)) * samples]) if per_sample else gens
            wave = np.zeros((0, 0), dtype=np.int16)
            if hi > lo:
                rows = (lo * samples, hi * samples, len(batch) * samples) if world > 1 else None
                with torch.no_grad():
                    latents = self.model.inference(batch[lo:hi], self.scheduler, steps, guidance, samples,
                                                   disable_progress=disable_progress, generator=g, noise_rows=rows, **kw)
                    wave = self._decode(latents)
            elif kw.get("latents") is None and kw.get("noises") is None:
                self.model.advance_rng(len(batch) * samples, self.scheduler, steps, g,
                                       kw.get("latent_shape", LATENT_HW))
            if world > 1:
                wave = parallel.allgather_waves(wave, self.device)
            outputs += [item for item in wave]
        if samples == 1:
            return outputs
        return list(self.chunks(outputs, samples))
