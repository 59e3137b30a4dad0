"""DDPM / DDIM / multistep DPM-Solver schedulers with the reference's interface; each update runs in one fused CUDA kernel.

Mirrors diffusers' DDPMScheduler / DDIMScheduler as Tango uses them
(/root/reference/mustango/diffusers/src/diffusers/schedulers/scheduling_ddpm.py:122-349,
scheduling_ddim.py:132-359; call sites models.py:224-249, tango.py:36): `set_timesteps`, `timesteps`,
`init_noise_sigma`, `order`, `scale_model_input`, `step(...).prev_sample`, `config`.

All per-step scalars are computed on the host with the reference's own fp32 torch ops (same association order),
packed into a [num_steps, 10] coefficient table and shipped to the device once per `set_timesteps`; the kernel
(tng_sched_step) then evaluates  x0 = (c0*s + c1*v)/c9, prev = c2*x0 + c3*s + c7*(c5*s + c6*v) + c4*noise  with
un-fused multiplies/adds, which reproduces the reference CPU arithmetic bit for bit and removes the two host syncs
per step of the reference (SURVEY.md §1).

DPMSolverMultistepScheduler (scheduling_dpmsolver_multistep.py) keeps the converted model outputs of the last two steps
in a device ring and runs tng_sched_multistep: its per-step scalars form a [num_steps, 11] table built the same way,
and the order each step uses follows the reference's `lower_order_nums` / `lower_order_final` state machine.

Every scheduler exposes `fused_step(i, ...)`: the CFG combine + update + next-UNet-input packing of step i of the
current grid, the one launch per step of AudioDiffusion.inference.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import numpy as np
import torch

from . import lib as L

# stabilityai/stable-diffusion-2-1 `scheduler/scheduler_config.json` — what Tango loads (tango.py:36, models.py:80-81).
# The JSON is not in the reference tree (SURVEY.md F6); these are its published values and every field can be overridden.
SD21_SCHEDULER_CONFIG = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012,
                             beta_schedule="scaled_linear", prediction_type="v_prediction", clip_sample=False,
                             set_alpha_to_one=False, steps_offset=1, skip_prk_steps=True, trained_betas=None)

NCOEF = 10


class SchedulerOutput(SimpleNamespace):
    pass


class _Config(dict):
    __getattr__ = dict.__getitem__


def _betas(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas=None):
    if trained_betas is not None:
        return torch.tensor(trained_betas, dtype=torch.float32)
    if beta_schedule == "linear":
        return torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    if beta_schedule == "scaled_linear":
        return torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    raise NotImplementedError(f"{beta_schedule} is not implemented")


class _SchedulerBase:
    order = 1

    def __init__(self, **cfg):
        self.config = _Config(cfg)
        self.betas = _betas(cfg["num_train_timesteps"], cfg["beta_start"], cfg["beta_end"], cfg["beta_schedule"],
                            cfg.get("trained_betas"))
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.init_noise_sigma = 1.0
        self.num_inference_steps: Optional[int] = None
        self.timesteps = torch.from_numpy(np.arange(0, cfg["num_train_timesteps"])[::-1].copy().astype(np.int64))
        self._coef_host: Optional[torch.Tensor] = None   # [num_steps, NCOEF] fp32 (CPU)
        self._coef_dev: Optional[torch.Tensor] = None
        self._t_index: dict = {}

    @classmethod
    def from_pretrained(cls, name: str = "stabilityai/stable-diffusion-2-1", subfolder: str = "scheduler", **overrides):
        """The reference downloads the SD-2.1 scheduler JSON from the hub (tango.py:36, models.py:80-81). Offline:
        a local directory is read (`<name>/<subfolder>/scheduler_config.json` or `<name>/scheduler_config.json`);
        `stabilityai/stable-diffusion-2-1` (or None) maps to its published values; any other name is refused rather
        than silently sampled with the wrong betas / prediction type."""
        import json
        import os
        base = dict(SD21_SCHEDULER_CONFIG)
        if name is not None and os.path.isdir(str(name)):
            for cand in (os.path.join(name, subfolder or "", "scheduler_config.json"), os.path.join(name, "scheduler_config.json")):
                if os.path.exists(cand):
                    with open(cand) as f:
                        base.update({k: v for k, v in json.load(f).items() if not k.startswith("_")})
                    break
            else:
                raise FileNotFoundError(f"no scheduler_config.json under '{name}'")
        elif name not in (None, "stabilityai/stable-diffusion-2-1"):
            raise ValueError(f"scheduler '{name}' is not reachable offline: pass a local directory holding its "
                             "scheduler_config.json (only stabilityai/stable-diffusion-2-1 is built in)")
        base.update(overrides)
        return cls(**{k: v for k, v in base.items() if k in cls._ACCEPTED})

    @classmethod
    def from_config(cls, config=None, **overrides):
        """diffusers' way to swap samplers: `DPMSolverMultistepScheduler.from_config(tango.scheduler.config)`. Keys
        this class does not take (e.g. DDIM's steps_offset) are ignored; keyword arguments override the config."""
        base = dict(config or {})
        base.update(overrides)
        return cls(**{k: v for k, v in base.items() if k in cls._ACCEPTED})

    def __len__(self):
        return self.config["num_train_timesteps"]

    def scale_model_input(self, sample, timestep=None):
        return sample

    # ---------------------------------------------------------------------------------------------------------
    def _grid(self, n: int) -> np.ndarray:
        T = self.config["num_train_timesteps"]
        if n > T:
            raise ValueError(
                f"`num_inference_steps`: {n} cannot be larger than `self.config.train_timesteps`: {T} as the unet"
                f" model trained with this scheduler can only handle maximal {T} timesteps.")
        ratio = T // n
        return (np.arange(0, n) * ratio).round()[::-1].copy().astype(np.int64)

    def _finish_set_timesteps(self, device):
        self._t_list = [int(t) for t in self.timesteps.tolist()]
        key = tuple(self._t_list)
        cache = self.__dict__.setdefault("_table_cache", {})
        if key not in cache:   # ~40 tiny fp32 torch ops per step: computed once per grid, reused by later calls
            cache[key] = torch.stack([self._coefficients(t) for t in self._t_list]).contiguous()
        self._coef_host = cache[key]
        self._t_index = {t: i for i, t in enumerate(self._t_list)}
        self._coef_dev = None
        if device is not None:
            self.timesteps = self.timesteps.to(device)
            if torch.device(device).type == "cuda":
                self._coef_dev = self._coef_host.to(device)

    def timestep_at(self, i: int) -> int:
        """Host copy of timesteps[i] (no device sync)."""
        return self._t_list[i]

    def coefficient_table(self, device=None) -> torch.Tensor:
        """[num_steps, 10] fp32 table (row i belongs to timesteps[i])."""
        if self._coef_host is None:
            self._finish_set_timesteps(None)
        if device is None:
            return self._coef_host
        if self._coef_dev is None or self._coef_dev.device != torch.device(device):
            self._coef_dev = self._coef_host.to(device)
        return self._coef_dev

    def _row(self, timestep) -> int:
        t = int(timestep)
        if self._coef_host is None or t not in self._t_index:
            # arbitrary timestep outside the current grid (the reference allows it): one-row table
            self._coef_host = self._coefficients(t)[None].contiguous()
            self._t_index = {t: 0}
            self._coef_dev = None
        return self._t_index[t]

    def fused_step(self, i: int, model_out, cfg, guidance, sample, noise, x_in, *, B, Cc, HW, split_off=0):
        """Step i of the current grid inside AudioDiffusion.inference: CFG combine of the channels-last UNet output,
        the update of `sample` in place and the packing of the next bf16 UNet input `x_in`, in one launch."""
        L.sched_step(model_out, cfg, guidance, sample, noise, self.coefficient_table(sample.device)[i], sample, x_in,
                     B=B, Cc=Cc, HW=HW, split_off=split_off)

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, generator=None,
             variance_noise: Optional[torch.Tensor] = None, return_dict: bool = True, **_unused):
        """x_t -> x_{t-1} for NCHW fp32 CUDA tensors (reference layout). Noise comes from the torch RNG exactly as
        in the reference (randn of model_output's shape when t > 0) unless `variance_noise` is given."""
        L.require_cuda(model_output)   # no CPU fallback
        i = self._row(timestep)
        coef = self.coefficient_table(sample.device)[i]
        B, Cc, H, W = sample.shape
        noise = None
        if self._needs_noise(int(timestep)):
            noise = variance_noise
            if noise is None:
                noise = torch.randn(model_output.shape, generator=generator, device=model_output.device,
                                    dtype=model_output.dtype)
            noise = noise.contiguous().float()
        mo = model_output.float().permute(0, 2, 3, 1).contiguous().view(B * H * W, Cc)  # channels-last rows
        prev = torch.empty_like(sample, dtype=torch.float32)
        L.sched_step(mo, False, 1.0, sample.contiguous().float(), noise, coef.contiguous(), prev, None, B=B, Cc=Cc,
                     HW=H * W)
        if not return_dict:
            return (prev,)
        return SchedulerOutput(prev_sample=prev)


class DDPMScheduler(_SchedulerBase):
    _ACCEPTED = ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule", "trained_betas", "variance_type",
                 "clip_sample", "prediction_type", "clip_sample_range")

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, variance_type="fixed_small", clip_sample=True, prediction_type="epsilon",
                 clip_sample_range=1.0):
        if variance_type != "fixed_small":
            raise NotImplementedError("only variance_type='fixed_small' (Tango's) is implemented")
        super().__init__(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                         beta_schedule=beta_schedule, trained_betas=trained_betas, variance_type=variance_type,
                         clip_sample=clip_sample, prediction_type=prediction_type,
                         clip_sample_range=clip_sample_range)
        self.one = torch.tensor(1.0)
        self.variance_type = variance_type

    def set_timesteps(self, num_inference_steps: int, device=None):
        """scheduling_ddpm.py:184-204: t_i = (i * (T // N)) reversed, int64 (no steps_offset in this version)."""
        self.timesteps = torch.from_numpy(self._grid(num_inference_steps))
        self.num_inference_steps = num_inference_steps
        self._finish_set_timesteps(device)

    def _needs_noise(self, t: int) -> bool:
        return t > 0

    def _coefficients(self, t: int) -> torch.Tensor:
        """scheduling_ddpm.py:283-344 scalar arithmetic, same fp32 torch ops in the same order."""
        cfg = self.config
        n = self.num_inference_steps if self.num_inference_steps else cfg["num_train_timesteps"]
        prev_t = t - cfg["num_train_timesteps"] // n
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.one
        b_t = 1 - a_t
        b_prev = 1 - a_prev
        cur_alpha = a_t / a_prev
        cur_beta = 1 - cur_alpha
        one, zero = torch.tensor(1.0), torch.tensor(0.0)
        if cfg["prediction_type"] == "epsilon":
            c_x0_s, c_x0_m, c_div = one, -(b_t ** 0.5), a_t ** 0.5
        elif cfg["prediction_type"] == "sample":
            c_x0_s, c_x0_m, c_div = zero, one, one
        elif cfg["prediction_type"] == "v_prediction":
            c_x0_s, c_x0_m, c_div = a_t ** 0.5, -(b_t ** 0.5), one
        else:
            raise ValueError(f"prediction_type given as {cfg['prediction_type']} must be one of `epsilon`, `sample` or"
                             " `v_prediction`  for the DDPMScheduler.")
        c_prev_x0 = (a_prev ** 0.5 * cur_beta) / b_t
        c_prev_s = cur_alpha ** 0.5 * b_prev / b_t
        c_noise = zero
        if t > 0:
            var = (1 - a_prev) / (1 - a_t) * cur_beta   # _get_variance :206-224
            var = torch.clamp(var, min=1e-20)
            c_noise = var ** 0.5
        clip = torch.tensor(float(cfg["clip_sample_range"]) if cfg["clip_sample"] else 0.0)
        return torch.stack([c_x0_s, c_x0_m, c_prev_x0, c_prev_s, c_noise, zero, zero, zero, clip, c_div]).float()


class DDIMScheduler(_SchedulerBase):
    _ACCEPTED = ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule", "trained_betas", "clip_sample",
                 "set_alpha_to_one", "steps_offset", "prediction_type", "clip_sample_range")

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, clip_sample=True, set_alpha_to_one=True, steps_offset=0,
                 prediction_type="epsilon", clip_sample_range=1.0):
        super().__init__(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                         beta_schedule=beta_schedule, trained_betas=trained_betas, clip_sample=clip_sample,
                         set_alpha_to_one=set_alpha_to_one, steps_offset=steps_offset,
                         prediction_type=prediction_type, clip_sample_range=clip_sample_range)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]

    def set_timesteps(self, num_inference_steps: int, device=None):
        """scheduling_ddim.py:214-236: same grid as DDPM plus steps_offset."""
        self.timesteps = torch.from_numpy(self._grid(num_inference_steps)) + self.config["steps_offset"]
        self.num_inference_steps = num_inference_steps
        self._finish_set_timesteps(device)

    def _needs_noise(self, t: int) -> bool:
        return False  # eta = 0 (deterministic DDIM)

    def _coefficients(self, t: int) -> torch.Tensor:
        """scheduling_ddim.py:292-354 with eta = 0."""
        cfg = self.config
        if self.num_inference_steps is None:
            raise ValueError("Number of inference steps is 'None', you need to run 'set_timesteps' after creating the"
                             " scheduler")
        prev_t = t - cfg["num_train_timesteps"] // self.num_inference_steps
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.final_alpha_cumprod
        b_t = 1 - a_t
        one, zero = torch.tensor(1.0), torch.tensor(0.0)
        if cfg["prediction_type"] == "epsilon":
            c_x0_s, c_x0_m, c_div = one, -(b_t ** 0.5), a_t ** 0.5
            c_eps_s, c_eps_m = zero, one
        elif cfg["prediction_type"] == "v_prediction":
            c_x0_s, c_x0_m, c_div = a_t ** 0.5, -(b_t ** 0.5), one
            c_eps_s, c_eps_m = b_t ** 0.5, a_t ** 0.5
        else:
            raise ValueError(f"prediction_type given as {cfg['prediction_type']} must be one of `epsilon` or"
                             " `v_prediction` for the fused DDIM step")
        b_prev = 1 - a_prev
        variance = (b_prev / b_t) * (1 - a_t / a_prev)
        std = 0.0 * variance ** 0.5
        c_prev_eps = (1 - a_prev - std ** 2) ** 0.5
        c_prev_x0 = a_prev ** 0.5
        clip = torch.tensor(float(cfg["clip_sample_range"]) if cfg["clip_sample"] else 0.0)
        return torch.stack([c_x0_s, c_x0_m, c_prev_x0, zero, zero, c_eps_s, c_eps_m, c_prev_eps, clip,
                            c_div]).float()


class DPMSolverMultistepScheduler(_SchedulerBase):
    """Multistep DPM-Solver / DPM-Solver++ (scheduling_dpmsolver_multistep.py): same constructor, defaults, `config`,
    timestep grid and stateful `step`. With CFG, `algorithm_type="dpmsolver++"` and `solver_order=2` (DPM-Solver++ 2M)
    is the usual choice for 10-25 steps.

    Coefficient row {c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4} of tng_sched_multistep, from the reference's fp32
    torch ops in its order (the reference's `A - k*D` terms become `A + (-k)*D`, which is exact):
      convert_model_output   m0 = (c_s * s + c_m * v) / c_div
      first order            x = k_s * s + k0 * m0
      second order           x = (k_s * s + k0 * m0) + k1 * (a1 * (m0 - m1))
      third order            E0 = a1 (m0 - m1), E1 = a2 (m1 - m2): x = ((...) + k1 (E0 + a3 (E0 - E1))) + k2 (a4 (E0 - E1))
    Not implemented (refused): dynamic thresholding (a per-sample quantile; the reference calls it unsuitable for latent
    models) and the squaredcos_cap_v2 beta schedule."""

    _ACCEPTED = ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule", "trained_betas", "solver_order",
                 "prediction_type", "thresholding", "dynamic_thresholding_ratio", "sample_max_value", "algorithm_type",
                 "solver_type", "lower_order_final")

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, solver_order=2, prediction_type="epsilon", thresholding=False,
                 dynamic_thresholding_ratio=0.995, sample_max_value=1.0, algorithm_type="dpmsolver++",
                 solver_type="midpoint", lower_order_final=True):
        if thresholding:
            raise NotImplementedError("thresholding=True (dynamic thresholding) is not implemented: it needs a "
                                      "per-sample quantile and is unsuitable for latent diffusion models")
        # the reference's remaps (its __init__): deis -> dpmsolver++, logrho / bh1 / bh2 -> midpoint
        if algorithm_type not in ("dpmsolver", "dpmsolver++"):
            if algorithm_type != "deis":
                raise NotImplementedError(f"{algorithm_type} is not implemented for {self.__class__}")
            algorithm_type = "dpmsolver++"
        if solver_type not in ("midpoint", "heun"):
            if solver_type not in ("logrho", "bh1", "bh2"):
                raise NotImplementedError(f"{solver_type} is not implemented for {self.__class__}")
            solver_type = "midpoint"
        if solver_order not in (1, 2, 3):
            raise ValueError(f"solver_order must be 1, 2 or 3, got {solver_order}")
        if prediction_type not in ("epsilon", "sample", "v_prediction"):
            raise ValueError(f"prediction_type given as {prediction_type} must be one of `epsilon`, `sample`, or"
                             " `v_prediction` for the DPMSolverMultistepScheduler.")
        super().__init__(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                         beta_schedule=beta_schedule, trained_betas=trained_betas, solver_order=solver_order,
                         prediction_type=prediction_type, thresholding=thresholding,
                         dynamic_thresholding_ratio=dynamic_thresholding_ratio, sample_max_value=sample_max_value,
                         algorithm_type=algorithm_type, solver_type=solver_type, lower_order_final=lower_order_final)
        self.alpha_t = torch.sqrt(self.alphas_cumprod)
        self.sigma_t = torch.sqrt(1 - self.alphas_cumprod)
        self.lambda_t = torch.log(self.alpha_t) - torch.log(self.sigma_t)
        self.timesteps = torch.from_numpy(
            np.linspace(0, num_train_timesteps - 1, num_train_timesteps, dtype=np.float32)[::-1].copy())
        self._orders: list = []
        self._extra_rows: dict = {}
        self._ring: Optional[list] = None
        self._reset_history()

    def _reset_history(self):
        """Forget the previous steps' model outputs (the reference's `model_outputs = [None] * order` and
        `lower_order_nums = 0`); the ring buffers themselves are reused."""
        self.lower_order_nums = 0
        self._ring_pos = 0

    def set_timesteps(self, num_inference_steps: int, device=None):
        """linspace(0, T - 1, N + 1).round() reversed, last entry dropped: starts at T - 1, no steps_offset."""
        T = self.config["num_train_timesteps"]
        self.num_inference_steps = num_inference_steps
        self.timesteps = torch.from_numpy(
            np.linspace(0, T - 1, num_inference_steps + 1).round()[::-1][:-1].copy().astype(np.int64))
        self._finish_set_timesteps(device)
        self._reset_history()

    def _finish_set_timesteps(self, device):
        self._t_list = [int(t) for t in self.timesteps.tolist()]
        key = (tuple(self._t_list), "orders")
        cache = self.__dict__.setdefault("_table_cache", {})
        if key not in cache:
            orders = self._fresh_orders(len(self._t_list))
            rows = [self._coefficients(t, i, o) for i, (t, o) in enumerate(zip(self._t_list, orders))]
            cache[key] = (torch.stack(rows).contiguous(), orders)
        self._coef_host, self._orders = cache[key]
        self._t_index = {t: i for i, t in enumerate(self._t_list)}
        self._coef_dev = None
        self._extra_rows = {}
        if device is not None:
            self.timesteps = self.timesteps.to(device)
            if torch.device(device).type == "cuda":
                self._coef_dev = self._coef_host.to(device)

    def _needs_noise(self, t: int) -> bool:
        return False

    @property
    def orders(self) -> list:
        """Solver order of each step of a loop started right after set_timesteps (row i of coefficient_table)."""
        return list(self._orders)

    def _order(self, i: int, n: int, lower_order_nums: int) -> int:
        """The reference's choice in `step`: lower orders while the history fills up, and for the last two steps of a
        grid shorter than 15 when lower_order_final is set."""
        cfg = self.config
        lof = cfg["lower_order_final"] and n < 15
        if cfg["solver_order"] == 1 or lower_order_nums < 1 or (lof and i == n - 1):
            return 1
        if cfg["solver_order"] == 2 or lower_order_nums < 2 or (lof and i == n - 2):
            return 2
        return 3

    def _fresh_orders(self, n: int) -> list:
        return [self._order(i, n, min(i, self.config["solver_order"])) for i in range(n)]

    def _coefficients(self, t: int, i: int, order: int) -> torch.Tensor:
        """Step i of the grid at (model) timestep t with the given order: scheduling_dpmsolver_multistep.py
        convert_model_output and the first / second / third order updates, same fp32 torch ops in the same order."""
        cfg = self.config
        ts = self._t_list
        n = len(ts)
        pp = cfg["algorithm_type"] == "dpmsolver++"
        a, sg, lam = self.alpha_t, self.sigma_t, self.lambda_t
        one, zero = torch.tensor(1.0), torch.tensor(0.0)
        pred = cfg["prediction_type"]
        if pp:
            c_s, c_m, c_div = {"epsilon": (one, -sg[t], a[t]), "sample": (zero, one, one),
                               "v_prediction": (a[t], -sg[t], one)}[pred]
        else:
            c_s, c_m, c_div = {"epsilon": (zero, one, one), "sample": (one, -a[t], sg[t]),
                               "v_prediction": (sg[t], a[t], one)}[pred]
        p = 0 if i == n - 1 else ts[i + 1]
        h = lam[p] - lam[t]
        if pp:
            k_s = sg[p] / sg[t]
            em1 = torch.exp(-h) - 1.0
            k0 = -(a[p] * em1)
        else:
            k_s = a[p] / a[t]
            em1 = torch.exp(h) - 1.0
            k0 = -(sg[p] * em1)
        k1 = k2 = a1 = a2 = a3 = a4 = zero
        if order == 2:
            r0 = (lam[t] - lam[ts[i - 1]]) / h
            a1 = 1.0 / r0
            if cfg["solver_type"] == "midpoint":
                k1 = -(0.5 * (a[p] * em1)) if pp else -(0.5 * (sg[p] * em1))
            else:
                k1 = a[p] * (em1 / h + 1.0) if pp else -(sg[p] * (em1 / h - 1.0))
        elif order == 3:
            s1, s2 = ts[i - 1], ts[i - 2]
            r0, r1 = (lam[t] - lam[s1]) / h, (lam[s1] - lam[s2]) / h
            a1, a2, a3, a4 = 1.0 / r0, 1.0 / r1, r0 / (r0 + r1), 1.0 / (r0 + r1)
            if pp:
                k1 = a[p] * (em1 / h + 1.0)
                k2 = -(a[p] * ((torch.exp(-h) - 1.0 + h) / h ** 2 - 0.5))
            else:
                k1 = -(sg[p] * (em1 / h - 1.0))
                k2 = -(sg[p] * ((torch.exp(h) - 1.0 - h) / h ** 2 - 0.5))
        return torch.stack([c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4]).float()

    def coefficient_table(self, device=None) -> torch.Tensor:
        """[num_steps, 11] fp32 table: row i is step i of a loop started right after set_timesteps (orders: `orders`)."""
        if self._coef_host is None:
            raise ValueError("Number of inference steps is 'None', you need to run 'set_timesteps' after creating the"
                             " scheduler")
        return super().coefficient_table(device)

    def _row(self, i: int, t: int, order: int, device) -> torch.Tensor:
        """Coefficient row for step i at timestep t with this order: the table row when the step is the one a fresh
        loop takes, otherwise (a timestep outside the grid, a reused history) computed once and cached."""
        if t == self._t_list[i] and order == self._orders[i]:
            return self.coefficient_table(device)[i]
        key = (i, t, order, str(device))
        row = self._extra_rows.get(key)
        if row is None:
            row = self._extra_rows[key] = self._coefficients(t, i, order).to(device)
        return row

    def _launch(self, i, t, model_out, cfg, guidance, sample, prev, x_in, *, B, Cc, HW, split_off=0):
        """One tng_sched_multistep: advances the history ring and the reference's `lower_order_nums`."""
        n = len(self._t_list)
        order = self._order(i, n, self.lower_order_nums)
        shape = (B, Cc, HW)
        if (self._ring is None or self._ring[0].shape != shape or self._ring[0].device != sample.device):
            self._ring = [torch.empty(shape, device=sample.device, dtype=torch.float32) for _ in range(3)]
        pos = self._ring_pos
        new = (pos + 1) % 3
        m1 = self._ring[pos] if order >= 2 else None
        m2 = self._ring[(pos + 2) % 3] if order >= 3 else None
        L.sched_multistep(model_out, cfg, guidance, sample, m1, m2, self._row(i, t, order, sample.device), order,
                          self._ring[new], prev, x_in, B=B, Cc=Cc, HW=HW, split_off=split_off)
        self._ring_pos = new
        if self.lower_order_nums < self.config["solver_order"]:
            self.lower_order_nums += 1

    def fused_step(self, i: int, model_out, cfg, guidance, sample, noise, x_in, *, B, Cc, HW, split_off=0):
        if noise is not None:
            raise ValueError("DPMSolverMultistepScheduler draws no per-step noise")
        self._launch(i, self._t_list[i], model_out, cfg, guidance, sample, sample, x_in, B=B, Cc=Cc, HW=HW,
                     split_off=split_off)

    def _step_index(self, timestep):
        """(index, timestep) without reading device memory: a view into `self.timesteps` (what iterating it yields)
        is located by its storage offset; any other value is looked up on the host. A timestep outside the grid maps
        to the last index, as in the reference."""
        if (isinstance(timestep, torch.Tensor) and timestep.numel() == 1 and isinstance(self.timesteps, torch.Tensor)
                and timestep.device == self.timesteps.device and timestep.dtype == self.timesteps.dtype
                and timestep.untyped_storage().data_ptr() == self.timesteps.untyped_storage().data_ptr()):
            i = timestep.storage_offset() - self.timesteps.storage_offset()
            if 0 <= i < len(self._t_list) and self.timesteps.stride(0) == 1:
                return i, self._t_list[i]
        t = int(timestep)
        return self._t_index.get(t, len(self._t_list) - 1), t

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, return_dict: bool = True, **_unused):
        """One multistep DPM-Solver step for NCHW tensors on a CUDA device (reference layout), stateful like the
        reference: the converted output is pushed into the history that set_timesteps resets."""
        if self.num_inference_steps is None:
            raise ValueError("Number of inference steps is 'None', you need to run 'set_timesteps' after creating the"
                             " scheduler")
        L.require_cuda(model_output, sample)   # no CPU fallback
        i, t = self._step_index(timestep)
        B, Cc, H, W = sample.shape
        mo = model_output.float().permute(0, 2, 3, 1).contiguous().view(B * H * W, Cc)  # channels-last rows
        prev = torch.empty_like(sample, dtype=torch.float32)
        self._launch(i, t, mo, False, 1.0, sample.contiguous().float(), prev, None, B=B, Cc=Cc, HW=H * W)
        if not return_dict:
            return (prev,)
        return SchedulerOutput(prev_sample=prev)

    def add_noise(self, original_samples: torch.Tensor, noise: torch.Tensor, timesteps: torch.Tensor) -> torch.Tensor:
        """Forward diffusion q(x_t | x_0) (training-time helper of the reference, plain torch: not on the sampling path)."""
        ac = self.alphas_cumprod.to(device=original_samples.device, dtype=original_samples.dtype)
        timesteps = timesteps.to(original_samples.device)
        sa = (ac[timesteps] ** 0.5).flatten()
        so = ((1 - ac[timesteps]) ** 0.5).flatten()
        while sa.dim() < original_samples.dim():
            sa, so = sa.unsqueeze(-1), so.unsqueeze(-1)
        return sa * original_samples + so * noise
