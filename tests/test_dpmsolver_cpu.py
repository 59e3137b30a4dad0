"""CPU: multistep DPM-Solver sampling (DPMSolverMultistepScheduler + tng_sched_multistep) without a GPU.

The oracle (oracle/dpmsolver.py) is pinned to the reference's own known answers and to tests/golden/dpmsolver.npz; the
product's timestep grids, coefficient table, order selection and history ring are run through the executable kernel
contract (tests/dpmsolver_spec.py) and compared with the oracle bit for bit. The kernel itself is checked against the
same contract on the GPU (test_dpmsolver_gpu.py). Nothing here is a CPU fallback of the product: the substitution
exists only under pytest's monkeypatch."""
import json
import os

import numpy as np
import pytest
import torch

import cabi_spec
import dpmsolver_spec as ds
from oracle.dpmsolver import OracleDPMSolverMultistep
from tango_b200 import lib as L
from tango_b200 import synth
from tango_b200.schedulers import DDIMScheduler, DDPMScheduler, DPMSolverMultistepScheduler

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CPU = torch.device("cpu")


@pytest.fixture
def spec_backend(monkeypatch):
    for name, fn in cabi_spec.SPEC.items():
        monkeypatch.setattr(L, name, fn)
    monkeypatch.setattr(L, "sched_multistep", ds.spec_sched_multistep)
    monkeypatch.setattr(L, "require_cuda_device", lambda device: None)
    monkeypatch.setattr(L, "require_cuda", lambda *ts: None)
    monkeypatch.setattr(L, "load", lambda *a, **k: None)


def _golden():
    return np.load(os.path.join(GOLD, "dpmsolver.npz"))


def _x0():
    return torch.from_numpy(_golden()["x0"])


# ------------------------------------------------------------------------------------------------------ the oracle
@pytest.mark.parametrize("pred,want", [("epsilon", 0.3301), ("v_prediction", 0.2251)])
def test_oracle_meets_reference_known_answers(pred, want):
    """The reference's own full-loop known answers for DPM-Solver++ 2M (linear betas, lower_order_final off)."""
    s = OracleDPMSolverMultistep(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                                 solver_order=2, prediction_type=pred, algorithm_type="dpmsolver++",
                                 solver_type="midpoint", lower_order_final=False)
    n = 4 * 3 * 8 * 8
    x = (torch.arange(n) / n).reshape(3, 8, 8, 4).permute(3, 0, 1, 2)
    x = ds.run_loop(s, x, 10, model=lambda x, t: x * t / (t + 1))
    assert round(x.abs().mean().item(), 4) == want


def test_oracle_matches_golden_bitwise():
    gd = _golden()
    n = 0
    for key, kw in ds.config_grid():
        x = ds.run_loop(OracleDPMSolverMultistep(**kw), _x0(), 10)
        assert torch.equal(x, torch.from_numpy(gd[f"loop_{key}"])), key
        n += 1
    assert n == 72


# ------------------------------------------------------------------------------------------------------ the product
@pytest.mark.parametrize("n", ds.GRID_STEPS)
def test_timestep_grid_matches_reference(n):
    s = DPMSolverMultistepScheduler(**ds.SD21_BETAS)
    s.set_timesteps(n)
    want = _golden()[f"timesteps_{n}"]
    assert s.timesteps.dtype == torch.int64 and np.array_equal(s.timesteps.numpy(), want)
    assert s.timesteps[0] == 999 and len(s.coefficient_table()) == n and len(s.orders) == n


def _orders_of_reference_loop(kw, n):
    """Order used at every step of a fresh loop, read from the oracle's state machine."""
    o = OracleDPMSolverMultistep(**kw)
    o.set_timesteps(n)
    used = []
    update = o.update
    o.update = lambda ms, ts, p, s: used.append(len(ms)) or update(ms, ts, p, s)
    ds.run_loop(o, _x0(), n)
    return used


@pytest.mark.parametrize("steps", [5, 10, 20, 25])
def test_table_orders_and_spec_match_oracle_over_config_grid(spec_backend, steps):
    """coefficient_table + orders + the kernel contract reproduce the reference loop with torch.equal, for every
    configuration; also `step` with the history ring, and (10 steps) the reference's own results."""
    gd = _golden()
    for key, kw in ds.config_grid():
        want = ds.run_loop(OracleDPMSolverMultistep(**kw), _x0(), steps)
        s = DPMSolverMultistepScheduler(**kw)
        s.set_timesteps(steps)
        assert s.orders == _orders_of_reference_loop(kw, steps), key
        # the table driven directly, as AudioDiffusion.inference does (fused_step), with an explicit ring
        x = _x0().clone()
        B, Cc, H, W = x.shape
        hist = []
        table = s.coefficient_table()
        assert table.shape == (steps, 11) and table.dtype == torch.float32
        for i, t in enumerate(s.timesteps.tolist()):
            mo = ds.model_fn(x, t).permute(0, 2, 3, 1).reshape(B * H * W, Cc)
            o = s.orders[i]
            m0, prev = torch.empty_like(x), torch.empty_like(x)
            ds.spec_sched_multistep(mo, False, 1.0, x, hist[-1] if o >= 2 else None, hist[-2] if o >= 3 else None,
                                    table[i], o, m0, prev, None, B=B, Cc=Cc, HW=H * W)
            hist.append(m0)
            x = prev
        assert torch.equal(x, want), key
        # the public, stateful `step`
        got = ds.run_loop(s, _x0(), steps)
        assert torch.equal(got, want), key
        if steps == 10:
            assert torch.equal(got, torch.from_numpy(gd[f"loop_{key}"])), key


def test_step_reuse_timestep_outside_grid_and_ring_reset(spec_backend):
    """The reference's stateful semantics: a second loop on the same object after set_timesteps starts from an empty
    history; without set_timesteps it keeps the history (and the higher order) of the first loop; a timestep outside
    the grid is treated as the last step."""
    kw = dict(ds.SD21_BETAS, solver_order=3, prediction_type="v_prediction", solver_type="heun")
    s, o = DPMSolverMultistepScheduler(**kw), OracleDPMSolverMultistep(**kw)
    for _ in range(2):
        assert torch.equal(ds.run_loop(s, _x0(), 10), ds.run_loop(o, _x0(), 10))
    # continue both without set_timesteps: history carried over, same as the reference
    x, y = _x0(), _x0()
    for t in s.timesteps.tolist()[:4] + [1]:      # 1 is not on the 10-step grid -> last index
        x = s.step(ds.model_fn(x, t), t, x).prev_sample
        y = o.step(ds.model_fn(y, t), t, y)
        assert torch.equal(x, y)
    assert s.lower_order_nums == 3


# ------------------------------------------------------------------------------------------------------ config
def test_config_loading_and_refusals(tmp_path):
    s = DPMSolverMultistepScheduler.from_pretrained("stabilityai/stable-diffusion-2-1", subfolder="scheduler")
    c = s.config
    assert (c.prediction_type, c.beta_schedule, c.solver_order, c.algorithm_type, c.solver_type) == \
        ("v_prediction", "scaled_linear", 2, "dpmsolver++", "midpoint")
    assert c.lower_order_final is True and s.init_noise_sigma == 1.0 and len(s) == 1000 and s.order == 1
    d = tmp_path / "snap" / "scheduler"
    d.mkdir(parents=True)
    (d / "scheduler_config.json").write_text(json.dumps({"_class_name": "DDIMScheduler", "beta_schedule": "linear",
                                                         "prediction_type": "epsilon", "steps_offset": 1}))
    s2 = DPMSolverMultistepScheduler.from_pretrained(str(tmp_path / "snap"), subfolder="scheduler", solver_order=3)
    assert (s2.config.beta_schedule, s2.config.prediction_type, s2.config.solver_order) == ("linear", "epsilon", 3)
    # from_config: the diffusers way to swap samplers; DDPM / DDIM gain it too
    ddpm = DDPMScheduler.from_pretrained(None)
    s3 = DPMSolverMultistepScheduler.from_config(ddpm.config)
    assert torch.equal(s3.alphas_cumprod, ddpm.alphas_cumprod) and s3.config.prediction_type == "v_prediction"
    assert DPMSolverMultistepScheduler.from_config(ddpm.config, solver_order=3).config.solver_order == 3
    ddim = DDIMScheduler.from_config(ddpm.config)
    assert ddim.config.prediction_type == "v_prediction" and ddim.config.steps_offset == 0
    assert DDPMScheduler.from_config(s3.config).config.beta_schedule == "scaled_linear"
    # refusals
    with pytest.raises(NotImplementedError):
        DPMSolverMultistepScheduler(thresholding=True)
    with pytest.raises(NotImplementedError):
        DPMSolverMultistepScheduler(beta_schedule="squaredcos_cap_v2")
    with pytest.raises(NotImplementedError):
        DPMSolverMultistepScheduler(algorithm_type="unipc")
    with pytest.raises(NotImplementedError):
        DPMSolverMultistepScheduler(solver_type="euler")
    with pytest.raises(ValueError):
        DPMSolverMultistepScheduler(prediction_type="x")
    with pytest.raises(ValueError):
        DPMSolverMultistepScheduler().step(torch.zeros(1), 999, torch.zeros(1))


@pytest.mark.parametrize("alg,st", [("deis", "midpoint"), ("dpmsolver++", "logrho"), ("deis", "bh1"),
                                    ("dpmsolver", "bh2")])
def test_remaps_like_the_reference(spec_backend, alg, st):
    kw = dict(ds.SD21_BETAS, algorithm_type=alg, solver_type=st, solver_order=3, prediction_type="epsilon")
    s = DPMSolverMultistepScheduler(**kw)
    want_alg = "dpmsolver++" if alg == "deis" else alg
    assert (s.config.algorithm_type, s.config.solver_type) == (want_alg, "midpoint")
    ref = DPMSolverMultistepScheduler(**dict(kw, algorithm_type=want_alg, solver_type="midpoint"))
    assert torch.equal(ds.run_loop(s, _x0(), 10), ds.run_loop(ref, _x0(), 10))
    assert torch.equal(ds.run_loop(s, _x0(), 10), ds.run_loop(OracleDPMSolverMultistep(**kw), _x0(), 10))


# ------------------------------------------------------------------------------------------------------ the loop
def test_advance_rng_consumes_one_latent_draw():
    from types import SimpleNamespace

    from tango_b200.pipeline import AudioDiffusion
    stub = SimpleNamespace(device=CPU, unet=SimpleNamespace(config={"in_channels": 8}))
    g = torch.Generator().manual_seed(11)
    AudioDiffusion.advance_rng(stub, 3, DPMSolverMultistepScheduler.from_pretrained(None), 20, g, (32, 16))
    ref = torch.Generator().manual_seed(11)
    torch.randn((3, 8, 32, 16), generator=ref)
    assert torch.equal(g.get_state(), ref.get_state())


class _NoEvent:
    def __init__(self, *a, **k):
        pass

    def record(self, *a, **k):
        pass

    def elapsed_time(self, other):
        return 0.0


@pytest.mark.parametrize("order,solver", [(2, "midpoint"), (3, "heun")])
def test_tiny_unet_cfg_loop_through_inference_matches_oracle(spec_backend, monkeypatch, order, solver):
    """AudioDiffusion.inference with DPM-Solver++ (CFG, per-step time embeddings of the DPM grid, fused CFG + multistep
    update) against the oracle pipeline on the same inputs, in split mode."""
    from oracle import pipeline as opipe
    from tango_b200.pipeline import AudioDiffusion
    monkeypatch.setattr(torch.cuda, "Event", _NoEvent)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(L, "launch_count", lambda: 0)
    cfg = synth.TINY_UNET_CONFIG
    sd = synth.synth_state_dict(synth.unet_param_shapes(cfg), seed=0)
    steps, guidance = 5, 3.0      # 5 steps: orders 1, 2, 3 (3M), and lower_order_final on the last two
    embeds, mask = synth.synth_conditioning(1, 9, cfg["cross_attention_dim"], seed=5, masked_tail=2)
    lat0, _ = synth.synth_noise(1, 1, shape=(8, 32, 16), seed=7)
    kw = dict(solver_order=order, solver_type=solver)
    want = opipe.inference(sd, cfg, OracleDPMSolverMultistep(**dict(ds.SD21_BETAS, prediction_type="v_prediction",
                                                                    **kw)), embeds, mask, steps, guidance, lat0)
    m = AudioDiffusion(unet_config=cfg, precision="split", use_cuda_graph=False).to(CPU)
    m.unet.load_state_dict(sd)
    sch = DPMSolverMultistepScheduler.from_pretrained(None, **kw)
    trace = []
    lat = m.inference(["x"], sch, steps, guidance, prompt_embeds=embeds, boolean_prompt_mask=mask, latents=lat0,
                      latent_shape=(32, 16), trace=trace)
    assert len(trace) == steps and sch.lower_order_nums == order
    err = float((lat.double() - want.double()).norm() / want.double().norm())
    assert err < 1e-4, err
