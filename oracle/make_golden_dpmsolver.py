"""Known answers for the multistep DPM-Solver scheduler (TEST INFRASTRUCTURE ONLY; needs /root/reference).

    python -m oracle.make_golden_dpmsolver [grid|config1]     (both by default; config1 takes ~10 min on 8 cores)

tests/golden/dpmsolver.npz — from the reference's unmodified DPMSolverMultistepScheduler
(mustango/diffusers/src/diffusers/schedulers/scheduling_dpmsolver_multistep.py):
  * `timesteps_<N>`: its timestep grid for every N in GRID_STEPS;
  * `x0` and `loop_<algorithm>_<solver>_o<order>_<prediction>_lof<0|1>`: the final sample of a 10-step loop with the
    deterministic stand-in model `model_fn` over the whole configuration grid (SD-2.1 betas).
  oracle/dpmsolver.py (OracleDPMSolverMultistep) is asserted bit-identical to every loop.

tests/golden/config1_dpmsolver.npz — the config-1 setup of oracle/make_golden_config1.py (same seeds and inputs: full
base UNet, 1 prompt, CFG 3, 10 steps, 256 x 16, fp32 CPU) run through the UNMODIFIED reference
`AudioDiffusion.inference` (models.py:210-257) with the reference's DPMSolverMultistepScheduler, twice: DPM-Solver++ 2M
midpoint and DPM-Solver++ 3M heun (SD-2.1 scheduler values). Final latents, timesteps and per-step latent norms are
stored; the oracle loop (oracle/pipeline.py + OracleDPMSolverMultistep) is asserted to agree within 5e-4.

What was checked and when goes to tests/golden/dpmsolver_manifest.json.
"""
from __future__ import annotations

import itertools
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import dpmsolver as odpm  # noqa: E402
from oracle import refshim  # noqa: E402
from oracle import schedulers as osched  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
GRID_STEPS = (1, 2, 3, 5, 10, 25, 50, 200, 999, 1000)
LOOP_STEPS = 10
SD21 = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
CONFIG1_RUNS = {"2m_midpoint": dict(solver_order=2, solver_type="midpoint"),
                "3m_heun": dict(solver_order=3, solver_type="heun")}


def grid_configs():
    """(key, scheduler kwargs) over algorithm x solver type x order x prediction type x lower_order_final."""
    for alg, st, order, pred, lof in itertools.product(("dpmsolver++", "dpmsolver"), ("midpoint", "heun"), (1, 2, 3),
                                                       ("epsilon", "v_prediction", "sample"), (True, False)):
        key = f"{alg.replace('++', 'pp')}_{st}_o{order}_{pred}_lof{int(lof)}"
        yield key, dict(SD21, algorithm_type=alg, solver_type=st, solver_order=order, prediction_type=pred,
                        lower_order_final=lof)


def model_fn(x, t):
    """Deterministic stand-in for the UNet: smooth in x, different at every timestep."""
    return torch.sin(x * 1.7 + int(t) * 0.01) * 0.9


def x0_tensor():
    return torch.randn(2, 4, 8, 4, generator=torch.Generator().manual_seed(0))


def loop(sch, x, steps=LOOP_STEPS):
    sch.set_timesteps(steps)
    for t in sch.timesteps:
        x = sch.step(model_fn(x, t), t, x)
        x = x.prev_sample if hasattr(x, "prev_sample") else x
    return x


def make_grid(manifest):
    R = _ref_class()
    out = {"x0": x0_tensor().numpy()}
    for n in GRID_STEPS:
        r = R(**SD21)
        r.set_timesteps(n)
        out[f"timesteps_{n}"] = r.timesteps.numpy()
    n_cfg = 0
    for key, kw in grid_configs():
        ref = loop(R(**kw), x0_tensor())
        orc = loop(odpm.OracleDPMSolverMultistep(**kw), x0_tensor())
        assert torch.equal(ref, orc), (key, float((ref - orc).abs().max()))
        out[f"loop_{key}"] = ref.numpy()
        n_cfg += 1
    path = os.path.join(GOLD, "dpmsolver.npz")
    np.savez_compressed(path, **out)
    manifest["checks"]["dpmsolver"] = {
        "configs": n_cfg, "loop_steps": LOOP_STEPS, "grid_steps": list(GRID_STEPS), "oracle_bit_exact": True,
        "what": "DPMSolverMultistepScheduler timestep grids and 10-step loops of a stand-in model over the "
                "algorithm x solver x order x prediction x lower_order_final grid"}
    print(f"tests/golden/dpmsolver.npz: {n_cfg} loops bit-exact ({os.path.getsize(path) / 1e3:.0f} kB)", flush=True)


def _ref_class():
    """The reference's DPMSolverMultistepScheduler, imported through the shim."""
    refshim.install()
    from diffusers.schedulers.scheduling_dpmsolver_multistep import DPMSolverMultistepScheduler
    return DPMSolverMultistepScheduler


def make_config1(manifest):
    from oracle import make_golden_config1 as c1
    from oracle import pipeline as opipe
    from tango_b200 import synth
    torch.set_grad_enabled(False)
    cfg, embeds, mask, lat0, _ = c1.inputs()
    sd = synth.synth_state_dict(synth.unet_param_shapes(cfg), seed=c1.SEEDS["weights"])
    U = refshim.unet_class()
    ref_unet = U.from_config(dict(cfg)).eval()
    ref_unet.load_state_dict(sd, strict=True)
    R = _ref_class()
    refmod = refshim.audio_diffusion_module()
    sc = dict(osched.SD21_CONFIG)

    class _Stub:
        pass

    out, checks = {}, {}
    for name, kw in CONFIG1_RUNS.items():
        skw = dict(SD21, prediction_type=sc["prediction_type"], algorithm_type="dpmsolver++", **kw)
        stub = _Stub()
        stub.unet = ref_unet
        stub.set_from = "random"
        stub.text_encoder = _Stub()
        stub.text_encoder.device = torch.device("cpu")
        stub.encode_text_classifier_free = lambda prompt, n: (embeds, mask)
        stub.prepare_latents = lambda bs, sch, ch, dt, dev: lat0 * sch.init_noise_sigma
        r = R(**skw)
        norms = []
        step0 = r.step

        def step(*a, _step0=step0, _norms=norms, **k):
            res = _step0(*a, **k)
            _norms.append(float(res.prev_sample.norm()))
            return res

        r.step = step
        t0 = time.time()
        lat_ref = refmod.AudioDiffusion.inference(stub, ["synthetic prompt"], r, c1.STEPS, c1.GUIDANCE, 1, True)
        t_ref = time.time() - t0
        trace = []
        t0 = time.time()
        lat_orc = opipe.inference(sd, cfg, odpm.OracleDPMSolverMultistep(**skw), embeds, mask, c1.STEPS, c1.GUIDANCE,
                                  lat0, None, trace=trace)
        t_orc = time.time() - t0
        d = c1.maxdiff(lat_ref, lat_orc)
        print(f"config-1 dpmsolver++ {name}: |lat| max {lat_ref.abs().max():.3f}, oracle-vs-reference max diff {d:.3e} "
              f"(reference {t_ref:.0f} s, oracle {t_orc:.0f} s)", flush=True)
        assert d < 5e-4, d
        assert len(norms) == c1.STEPS
        out[f"latents_{name}"] = lat_ref.numpy()
        out[f"timesteps_{name}"] = r.timesteps.numpy()
        out[f"step_norms_{name}"] = np.asarray(norms, dtype=np.float64)
        checks[name] = {"scheduler": skw, "latents_max_abs": d, "reference_s": round(t_ref, 1),
                        "oracle_s": round(t_orc, 1)}
    path = os.path.join(GOLD, "config1_dpmsolver.npz")
    np.savez_compressed(path, **out)
    manifest["checks"]["config1_dpmsolver"] = dict(
        checks, generated=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), seeds=c1.SEEDS, steps=c1.STEPS,
        guidance=c1.GUIDANCE, tokens=c1.TOKENS,
        what="config-1 (full base UNet, 1 prompt, CFG 3, 10 steps, fp32 CPU) through the unmodified reference loop "
             "with DPMSolverMultistepScheduler: DPM-Solver++ 2M midpoint and 3M heun")
    print(f"tests/golden/config1_dpmsolver.npz written ({os.path.getsize(path) / 1e6:.2f} MB)", flush=True)


def main(parts):
    mp = os.path.join(GOLD, "dpmsolver_manifest.json")
    manifest = json.load(open(mp)) if os.path.exists(mp) else {
        "what": "Provenance of the DPM-Solver known answers (written by oracle/make_golden_dpmsolver.py)", "checks": {}}
    manifest["reference"] = f"declare-lab/tango @ {refshim.REF} (diffusers fork 0.15.0.dev0)"
    manifest["torch"] = torch.__version__
    if "grid" in parts:
        make_grid(manifest)
    if "config1" in parts:
        make_config1(manifest)
    with open(mp, "w") as f:
        json.dump(manifest, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1:] or ["grid", "config1"])
