"""CPU restatement of DPMSolverMultistepScheduler (TEST INFRASTRUCTURE ONLY).

Follows /root/reference/mustango/diffusers/src/diffusers/schedulers/scheduling_dpmsolver_multistep.py operation by
operation in torch fp32 on the CPU, so the results are bit-identical to the reference run on CPU
(oracle/make_golden_dpmsolver.py asserts it over the whole configuration grid).
"""
from __future__ import annotations

import numpy as np
import torch

from .schedulers import make_betas


class OracleDPMSolverMultistep:
    """scheduling_dpmsolver_multistep.py (multistep DPM-Solver / DPM-Solver++, no thresholding) restated operation by
    operation: convert_model_output, the first / second / third order updates and the `lower_order_nums` /
    `lower_order_final` order selection of `step`."""

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 solver_order=2, prediction_type="epsilon", algorithm_type="dpmsolver++", solver_type="midpoint",
                 lower_order_final=True, **_ignored):
        self.T = num_train_timesteps
        self.betas = make_betas(num_train_timesteps, beta_start, beta_end, beta_schedule)
        self.alphas_cumprod = torch.cumprod(1.0 - self.betas, dim=0)
        self.alpha_t = torch.sqrt(self.alphas_cumprod)
        self.sigma_t = torch.sqrt(1 - self.alphas_cumprod)
        self.lambda_t = torch.log(self.alpha_t) - torch.log(self.sigma_t)
        self.init_noise_sigma = 1.0
        self.order_max, self.prediction_type = solver_order, prediction_type
        self.algorithm_type = "dpmsolver++" if algorithm_type == "deis" else algorithm_type
        self.solver_type = "midpoint" if solver_type in ("logrho", "bh1", "bh2") else solver_type
        self.lower_order_final = lower_order_final
        self.num_inference_steps = None

    def set_timesteps(self, n):
        self.num_inference_steps = n
        self.timesteps = torch.from_numpy(np.linspace(0, self.T - 1, n + 1).round()[::-1][:-1].copy().astype(np.int64))
        self.history = []
        self.lower_order_nums = 0

    def convert(self, v, t, s):
        a, sg = self.alpha_t[t], self.sigma_t[t]
        if self.algorithm_type == "dpmsolver++":
            if self.prediction_type == "epsilon":
                return (s - sg * v) / a
            if self.prediction_type == "sample":
                return v
            return a * s - sg * v
        if self.prediction_type == "epsilon":
            return v
        if self.prediction_type == "sample":
            return (s - a * v) / sg
        return a * v + sg * s

    def update(self, ms, ts, p, s):
        """Order len(ms) update from timesteps ts (oldest first) to p; ms: converted outputs, oldest first."""
        lam, a, sg = self.lambda_t, self.alpha_t, self.sigma_t
        s0 = ts[-1]
        h = lam[p] - lam[s0]
        pp = self.algorithm_type == "dpmsolver++"
        if pp:
            x = (sg[p] / sg[s0]) * s - (a[p] * (torch.exp(-h) - 1.0)) * ms[-1]
        else:
            x = (a[p] / a[s0]) * s - (sg[p] * (torch.exp(h) - 1.0)) * ms[-1]
        if len(ms) == 2:
            r0 = (lam[s0] - lam[ts[-2]]) / h
            d1 = (1.0 / r0) * (ms[-1] - ms[-2])
            if self.solver_type == "midpoint":
                k = (a[p] * (torch.exp(-h) - 1.0)) if pp else (sg[p] * (torch.exp(h) - 1.0))
                x = x - 0.5 * k * d1
            elif pp:
                x = x + (a[p] * ((torch.exp(-h) - 1.0) / h + 1.0)) * d1
            else:
                x = x - (sg[p] * ((torch.exp(h) - 1.0) / h - 1.0)) * d1
        elif len(ms) == 3:
            r0, r1 = (lam[s0] - lam[ts[-2]]) / h, (lam[ts[-2]] - lam[ts[-3]]) / h
            e0, e1 = (1.0 / r0) * (ms[-1] - ms[-2]), (1.0 / r1) * (ms[-2] - ms[-3])
            d1 = e0 + (r0 / (r0 + r1)) * (e0 - e1)
            d2 = (1.0 / (r0 + r1)) * (e0 - e1)
            if pp:
                x = x + (a[p] * ((torch.exp(-h) - 1.0) / h + 1.0)) * d1
                x = x - (a[p] * ((torch.exp(-h) - 1.0 + h) / h ** 2 - 0.5)) * d2
            else:
                x = x - (sg[p] * ((torch.exp(h) - 1.0) / h - 1.0)) * d1
                x = x - (sg[p] * ((torch.exp(h) - 1.0 - h) / h ** 2 - 0.5)) * d2
        return x

    def step(self, model_output, t, sample, noise=None):
        ts = [int(x) for x in self.timesteps]
        t = int(t)
        n = len(ts)
        i = ts.index(t) if t in ts else n - 1
        p = 0 if i == n - 1 else ts[i + 1]
        lof = self.lower_order_final and n < 15
        self.history = (self.history + [self.convert(model_output, t, sample)])[-self.order_max:]
        if self.order_max == 1 or self.lower_order_nums < 1 or (lof and i == n - 1):
            order = 1
        elif self.order_max == 2 or self.lower_order_nums < 2 or (lof and i == n - 2):
            order = 2
        else:
            order = 3
        grid = [ts[i - k] for k in range(order - 1, 0, -1)]   # negative indices wrap, as the reference's do
        x = self.update(self.history[-order:], grid + [t], p, sample)
        self.lower_order_nums = min(self.lower_order_nums + 1, self.order_max)
        return x
