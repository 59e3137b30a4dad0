"""Executable statement of `tng_sched_multistep` (TEST INFRASTRUCTURE ONLY), in the style of tests/cabi_spec.py: a few
lines of torch on the CPU that state the kernel's contract, so the multistep scheduler and the sampling loop can run
without a GPU (tests/test_dpmsolver_cpu.py) and the kernel can be compared with it bit for bit on one
(tests/test_dpmsolver_gpu.py). It mirrors the signature of tango_b200.lib.sched_multistep and is never imported by the
package."""
from __future__ import annotations

from cabi_spec import _store_bf16


def spec_sched_multistep(model_out, cfg, guidance, sample, m1, m2, coef, order, m0, prev, next_in, *, B, Cc, HW,
                         split_off=0):
    """CFG combine + multistep DPM-Solver update with coefficient row {c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4}
    (fp32 0-d tensors, so every product and sum rounds to fp32 on its own, as in the kernel) + packing of the next UNet
    input. model_out: channels-last rows [(2)B*HW, >=Cc]; sample / m1 / m2 / m0 / prev: NCHW fp32."""
    c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4 = [coef.reshape(-1)[i] for i in range(11)]
    s = sample.reshape(B, Cc, HW).float()
    mo = model_out[:, :Cc].float()
    if cfg:
        u, t = mo[:B * HW].reshape(B, HW, Cc), mo[B * HW:2 * B * HW].reshape(B, HW, Cc)
        v = u + guidance * (t - u)
    else:
        v = mo[:B * HW].reshape(B, HW, Cc)
    v = v.transpose(1, 2)
    x0 = (c_s * s + c_m * v) / c_div
    out = k_s * s + k0 * x0
    if order == 2:
        out = out + k1 * (a1 * (x0 - m1.reshape(B, Cc, HW)))
    elif order == 3:
        h1, h2 = m1.reshape(B, Cc, HW), m2.reshape(B, Cc, HW)
        e0, e1 = a1 * (x0 - h1), a2 * (h1 - h2)
        out = (out + k1 * (e0 + a3 * (e0 - e1))) + k2 * (a4 * (e0 - e1))
    m0.reshape(B, Cc, HW).copy_(x0)
    if prev is not None:
        prev.reshape(B, Cc, HW).copy_(out)
    if next_in is not None:
        rows = out.transpose(1, 2).reshape(B * HW, Cc)
        for r in range(2 if cfg else 1):
            _store_bf16(next_in[r * B * HW:(r + 1) * B * HW], rows, split_off)


# The configuration grid and stand-in model of tests/golden/dpmsolver.npz (oracle/make_golden_dpmsolver.py).
SD21_BETAS = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
GRID_STEPS = (1, 2, 3, 5, 10, 25, 50, 200, 999, 1000)


def config_grid():
    """(key, scheduler kwargs) over algorithm x solver type x order x prediction type x lower_order_final."""
    import itertools
    for alg, st, order, pred, lof in itertools.product(("dpmsolver++", "dpmsolver"), ("midpoint", "heun"), (1, 2, 3),
                                                       ("epsilon", "v_prediction", "sample"), (True, False)):
        key = f"{alg.replace('++', 'pp')}_{st}_o{order}_{pred}_lof{int(lof)}"
        yield key, dict(SD21_BETAS, algorithm_type=alg, solver_type=st, solver_order=order, prediction_type=pred,
                        lower_order_final=lof)


def model_fn(x, t):
    """Deterministic stand-in for the UNet: smooth in x, different at every timestep."""
    import torch
    return torch.sin(x * 1.7 + int(t) * 0.01) * 0.9


def run_loop(sch, x, steps, model=model_fn):
    """set_timesteps + one `step` per timestep, iterating `sch.timesteps` like AudioDiffusion.inference."""
    sch.set_timesteps(steps, **({"device": x.device} if x.is_cuda else {}))
    for t in sch.timesteps:
        x = sch.step(model(x, t), t, x)
        x = x.prev_sample if hasattr(x, "prev_sample") else x
    return x
