"""CPU: pin the oracle (oracle/*.py) against (a) the golden vectors generated from the REAL reference by
oracle/make_golden.py and (b) the known-answer constants of the diffusers fork's own tests
(mustango/diffusers/tests/test_layers_utils.py:92-117, schedulers/test_scheduler_ddpm.py:62-131,
schedulers/test_scheduler_ddim.py:46-54,94-122)."""
import os

import numpy as np
import pytest
import torch

from oracle import hifigan as ohifi
from oracle import pipeline as opipe
from oracle import schedulers as osched
from oracle import unet as ounet
from oracle import vae as ovae
from tango_b200 import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def gold(name):
    return np.load(os.path.join(GOLD, name))


def test_sinusoid_hardcoded():
    t = torch.arange(128)
    t1 = ounet.timestep_embedding(t, 64, flip_sin_to_cos=False, freq_shift=1)
    t2 = ounet.timestep_embedding(t, 64, flip_sin_to_cos=True, freq_shift=0)
    assert torch.allclose(t1[23:26, 47:50].flatten(),
                          torch.tensor([0.9646, 0.9804, 0.9892, 0.9615, 0.9787, 0.9882, 0.9582, 0.9769, 0.9872]), 1e-3)
    assert torch.allclose(t2[23:26, 47:50].flatten(),
                          torch.tensor([0.3019, 0.2280, 0.1716, 0.3146, 0.2377, 0.1790, 0.3272, 0.2474, 0.1864]), 1e-3)


def _dummy_sample_deter():
    # mustango/diffusers/tests/schedulers/test_schedulers.py:236-247
    n = 4 * 3 * 8 * 8
    s = torch.arange(n).reshape(3, 8, 8, 4) / n
    return s.permute(3, 0, 1, 2)


def _dummy_model(sample, t):
    return sample * t / (t + 1)


@pytest.mark.parametrize("pred,exp_sum,exp_mean", [("epsilon", 258.9606, 0.3372), ("v_prediction", 202.0296, 0.2631)])
def test_ddpm_full_loop_constants(pred, exp_sum, exp_mean):
    s = osched.OracleDDPM(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                          clip_sample=True, prediction_type=pred)
    sample = _dummy_sample_deter()
    g = torch.manual_seed(0)
    for t in reversed(range(1000)):
        res = _dummy_model(sample, t)
        noise = torch.randn(res.shape, generator=g) if t > 0 else None
        sample = s.step(res, t, sample, noise)
    assert abs(sample.abs().sum().item() - exp_sum) < 1e-2
    assert abs(sample.abs().mean().item() - exp_mean) < 1e-3


def test_ddpm_variance_constants():
    s = osched.OracleDDPM(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear")
    assert abs(float(s._get_variance(0)) - 0.0) < 1e-5
    assert abs(float(s._get_variance(487)) - 0.00979) < 1e-5
    assert abs(float(s._get_variance(999)) - 0.02) < 1e-5


def test_ddim_offset_grid_and_loops():
    s = osched.OracleDDIM(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                          steps_offset=1)
    s.set_timesteps(5)
    assert torch.equal(s.timesteps, torch.LongTensor([801, 601, 401, 201, 1]))
    for pred, es, em in (("epsilon", 172.0067, 0.223967), ("v_prediction", 52.5302, 0.0684)):
        s = osched.OracleDDIM(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                              clip_sample=True, prediction_type=pred)
        s.set_timesteps(10)
        x = _dummy_sample_deter()
        for t in s.timesteps:
            x = s.step(_dummy_model(x, t), t, x)
        assert abs(x.abs().sum().item() - es) < 1e-2
        assert abs(x.abs().mean().item() - em) < 1e-3


def test_scheduler_goldens_bit_exact():
    gd = gold("schedulers.npz")
    sc = osched.SD21_CONFIG
    for n in (10, 200):
        o = osched.OracleDDPM(**sc)
        o.set_timesteps(n)
        assert np.array_equal(o.timesteps.numpy(), gd[f"ddpm_timesteps_{n}"])
        oi = osched.OracleDDIM(**sc)
        oi.set_timesteps(n)
        assert np.array_equal(oi.timesteps.numpy(), gd[f"ddim_timesteps_{n}"])
    assert gd["ddpm_timesteps_200"][0] == 995 and gd["ddpm_timesteps_200"][-1] == 0
    assert gd["ddim_timesteps_200"][0] == 996 and gd["ddim_timesteps_200"][-1] == 1
    x0 = torch.from_numpy(gd["x0"])
    noises = torch.from_numpy(gd["noises"])
    for pred in ("v_prediction", "epsilon"):
        o = osched.OracleDDPM(**dict(sc, prediction_type=pred))
        o.set_timesteps(10)
        x = x0.clone()
        for i, t in enumerate(o.timesteps):
            x = o.step(torch.sin(x * 3.0 + float(t) / 1000), t, x, noises[i])
        assert np.array_equal(x.numpy(), gd[f"ddpm_loop_{pred}"])
        oi = osched.OracleDDIM(**dict(sc, prediction_type=pred))
        oi.set_timesteps(10)
        x = x0.clone()
        for t in oi.timesteps:
            x = oi.step(torch.sin(x * 3.0 + float(t) / 1000), t, x)
        assert np.array_equal(x.numpy(), gd[f"ddim_loop_{pred}"])


def test_tiny_unet_golden():
    gd = gold("tiny_unet.npz")
    cfg = synth.TINY_UNET_CONFIG
    sd = synth.synth_state_dict(synth.unet_param_shapes(cfg), seed=0)
    out = ounet.unet_forward(sd, cfg, torch.from_numpy(gd["sample"]), torch.tensor(int(gd["t"])),
                             torch.from_numpy(gd["ehs"]), torch.from_numpy(gd["mask"]))
    assert np.abs(out.numpy() - gd["out"]).max() < 5e-5
    out2 = ounet.unet_forward(sd, cfg, torch.from_numpy(gd["sample"]), 7, torch.from_numpy(gd["ehs"]), None)
    assert np.abs(out2.numpy() - gd["out_nomask_t7"]).max() < 5e-5


def test_tiny_vae_vocoder_golden():
    gd = gold("tiny_vae_vocoder.npz")
    vsd = synth.synth_state_dict(synth.vae_decoder_param_shapes(), seed=0)
    mel = ovae.decode_first_stage(vsd, torch.from_numpy(gd["z"]), synth.VAE_CONFIG["scale_factor"])
    assert np.abs(mel.numpy() - gd["mel"]).max() < 1e-4
    wav, wi = ohifi.decode_to_waveform(vsd, mel)
    assert np.abs(wav.numpy() - gd["wave"]).max() < 1e-4
    assert np.abs(wi.astype(np.int32) - gd["wave_i16"].astype(np.int32)).max() <= 2
    assert wi.dtype == np.int16 and wi.shape == (1, 5152)  # (32 mel frames -> 5*4*2*2*2*32 + tail)


def test_tiny_inference_golden():
    gd = gold("tiny_inference.npz")
    cfg = synth.TINY_UNET_CONFIG
    sd = synth.synth_state_dict(synth.unet_param_shapes(cfg), seed=0)
    o = osched.OracleDDPM(**osched.SD21_CONFIG)
    noises = [torch.from_numpy(n) for n in gd["noises"]]
    lat = opipe.inference(sd, cfg, o, torch.from_numpy(gd["embeds"]), torch.from_numpy(gd["mask"]), 4, 3.0,
                          torch.from_numpy(gd["lat0"]), noises)
    assert np.abs(lat.numpy() - gd["latents"]).max() < 2e-4


def test_tiny_t5_golden():
    """oracle/t5.py against outputs of transformers.T5EncoderModel (tests/golden/tiny_t5.npz, oracle/make_golden_t5.py)."""
    from oracle import t5 as ot5
    gd = gold("tiny_t5.npz")
    cfg = synth.TINY_T5_CONFIG
    assert cfg == ot5.TINY_T5_CONFIG
    sd = synth.synth_state_dict(synth.t5_encoder_param_shapes(cfg), seed=0)
    out = ot5.t5_encoder(sd, cfg, torch.from_numpy(gd["ids"]), torch.from_numpy(gd["mask"]))
    assert np.abs(out.numpy() - gd["out"]).max() < 2e-5
    out = ot5.t5_encoder(sd, cfg, torch.from_numpy(gd["ids_long"]), torch.from_numpy(gd["mask_long"]))
    assert np.abs(out.numpy() - gd["out_long"]).max() < 2e-5


def test_t5_bucket_known_answers():
    """Bucket layout of the bidirectional relative attention (32 buckets, max distance 128): exact offsets below 8,
    logarithmic bins above, positive offsets shifted by 16, saturation at |offset| >= 128."""
    from oracle import t5 as ot5
    rel = torch.tensor([0, -1, -7, -8, -15, -16, -127, -128, -1000, 1, 7, 8, 127, 128, 1000])
    b = ot5.relative_position_bucket(rel, 32, 128).tolist()
    assert b == [0, 1, 7, 8, 9, 10, 15, 15, 15, 17, 23, 24, 31, 31, 31]


def test_tiny_vae_encoder_golden():
    """oracle/vae.py:encode_first_stage against the reference AutoencoderKL.encode_first_stage posterior
    (tests/golden/tiny_vae_encoder.npz, oracle/make_golden_vae_encoder.py) — checker for the "next" row 2."""
    gd = gold("tiny_vae_encoder.npz")
    esd = synth.synth_state_dict(synth.vae_encoder_param_shapes(), seed=0)
    mean, std = ovae.encode_first_stage(esd, torch.from_numpy(gd["mel"]))
    assert mean.shape == (2, 8, 16, 16)
    assert np.abs(mean.numpy() - gd["mean"]).max() < 1e-5 and np.abs(std.numpy() - gd["std"]).max() < 1e-5


def test_tiny_stft_frontend_golden():
    """oracle/stft.py (waveform conditioning, windowed-DFT magnitude, mel projection, log compression, padding) against
    the reference's STFT / TacotronSTFT / torch_tools arithmetic (tests/golden/tiny_stft.npz, oracle/make_golden_stft.py)."""
    from oracle import stft as ostft
    gd = gold("tiny_stft.npz")
    FL, HOP, WIN, NMEL, target = (int(v) for v in gd["cfg"])
    basis = ostft.forward_basis(FL, WIN)
    assert basis.shape == (2 * (FL // 2 + 1), 1, FL)
    fb, lm, wav = ostft.wav_to_fbank([torch.from_numpy(gd["wave0"]), torch.from_numpy(gd["wave1"])], basis,
                                     torch.from_numpy(gd["mel_basis"]), target_length=target, filter_length=FL,
                                     hop_length=HOP)
    assert fb.shape == (2, target, NMEL) and lm.shape == (2, target, FL // 2)
    assert np.abs(wav.numpy() - gd["wav"]).max() < 1e-6
    assert np.abs(fb.numpy() - gd["fbank"]).max() < 1e-5 and np.abs(lm.numpy() - gd["log_mag"]).max() < 1e-5
    # DFT sanity: a pure tone at bin 8 puts its energy in magnitude bin 8
    t = torch.arange(FL * 4, dtype=torch.float32)
    mag = ostft.stft_magnitude(0.5 * torch.sin(2 * np.pi * 8 * t / FL)[None], basis, FL, HOP)
    assert int(mag[0, :, 5].argmax()) == 8


# Known-answer slices hard-coded in the diffusers fork's own block tests (mustango/diffusers/tests/test_layers_utils.py):
# ResnetBlock2D default :226-240, Upsample2D with conv :131-141, Downsample2D with conv / padding 1 :200-210,
# Transformer2DModel with cross attention :394-418. Each test seeds torch with 0, draws the input, then builds the module
# with default initialisation; oracle/make_golden_blocks.py stores those module weights (tests/golden/block_known_answers/).
BLOCK_KNOWN = {
    "resnet": [-1.9010, -0.2974, -0.8245, -1.3533, 0.8742, -0.9645, -2.0584, 1.3387, -0.4746],
    "upsample": [0.7145, 1.3773, 0.3492, 0.8448, 1.0839, -0.3341, 0.5956, 0.1250, -0.4841],
    "downsample": [0.9267, 0.5878, 0.3337, 1.2321, -0.1191, -0.3984, -0.7532, -0.0715, -0.3913],
    "transformer": [-0.2555, -0.8877, -2.4739, -2.2251, 1.2714, 0.0807, -0.4161, -1.6408, -0.0471],
}


def _seeded_input(gd, name, shape):
    torch.manual_seed(0)
    x = torch.randn(*shape)
    if abs(float(x.double().sum()) - float(gd[name + "_x_sum"])) > 1e-3:
        pytest.skip("torch CPU RNG stream differs from the build that wrote the fixture")
    return x


@pytest.mark.parametrize("name", sorted(BLOCK_KNOWN))
def test_oracle_blocks_meet_reference_known_answers(name):
    gd = gold(f"block_known_answers/{name}.npz")
    sd = {k[len(name) + 1:]: torch.from_numpy(gd[k]) for k in gd.files if k.startswith(name + ".")}
    if name == "resnet":
        x = _seeded_input(gd, name, (1, 32, 64, 64))
        sd = {"r." + k: v for k, v in sd.items()}
        y = ounet.resnet_block(sd, "r", x, torch.from_numpy(gd["resnet_temb"]), 32, 1e-6)   # ResnetBlock2D defaults
    elif name == "upsample":
        y = ounet.upsample2d({"u." + k: v for k, v in sd.items()}, "u", _seeded_input(gd, name, (1, 32, 32, 32)))
    elif name == "downsample":
        y = ounet.downsample2d({"d." + k: v for k, v in sd.items()}, "d", _seeded_input(gd, name, (1, 32, 64, 64)))
    else:
        # the test's block uses 1x1-conv projections (use_linear_projection=False): identical arithmetic to the linear
        # form the oracle restates (Tango's config), with the conv kernels viewed as matrices
        x = _seeded_input(gd, name, (1, 64, 64, 64))
        sd = {"t." + k: (v[:, :, 0, 0] if k in ("proj_in.weight", "proj_out.weight") else v) for k, v in sd.items()}
        y = ounet.transformer_2d(sd, "t", x, torch.from_numpy(gd["transformer_ctx"]), 2, 32, None)
    got = y[0, -1, -3:, -3:].flatten()
    assert torch.allclose(got, torch.tensor(BLOCK_KNOWN[name]), atol=1e-3), (name, got)


# Known-answer slices of the fork's UNet block tests (mustango/diffusers/tests/test_unet_2d_blocks.py, harness in
# test_unet_blocks_common.py:41-105): DownBlock2D :23-30, CrossAttnDownBlock2D :50-62, UNetMidBlock2DCrossAttn :168-179,
# UpBlock2D :200-211, CrossAttnUpBlock2D :226-241 — every block type of Tango's UNet configs. Compared at the tests' own
# tolerance (5e-3); the blocks are composed here from the oracle's resnet / transformer / resampling functions exactly as
# oracle/unet.py:unet_forward composes them.
UNET_BLOCK_KNOWN = {
    "DownBlock2D": [-0.0232, -0.9869, 0.8054, -0.0637, -0.1688, -1.4264, 0.4470, -1.3394, 0.0904],
    "CrossAttnDownBlock2D": [0.2440, -0.6953, -0.2140, -0.3874, 0.1966, 1.2077, 0.0441, -0.7718, 0.2800],
    "UNetMidBlock2DCrossAttn": [0.1879, 2.2653, 0.5987, 1.1568, -0.8454, -1.6109, -0.8919, 0.8306, 1.6758],
    "UpBlock2D": [-0.2041, -0.4165, -0.3022, 0.0041, -0.6628, -0.7053, 0.1928, -0.0325, 0.0523],
    "CrossAttnUpBlock2D": [-0.2796, -0.4364, -0.1067, -0.2693, 0.1894, 0.3869, -0.3470, 0.4584, 0.5091],
}


@pytest.mark.parametrize("name", sorted(UNET_BLOCK_KNOWN))
def test_oracle_unet_blocks_meet_reference_known_answers(name):
    gd = gold(f"block_known_answers/{name}.npz")
    sd = {k[len(name) + 1:]: torch.from_numpy(gd[k]) for k in gd.files if k.startswith(name + ".")}
    # the harness builds the attention blocks with 1x1-conv projections; same arithmetic as the linear form
    sd = {k: (v[:, :, 0, 0] if k.endswith(("proj_in.weight", "proj_out.weight")) and v.dim() == 4 else v)
          for k, v in sd.items()}
    g = torch.manual_seed(0)
    hs = torch.randn(4, 32, 32, 32, generator=g)
    temb = torch.randn(4, 128, generator=g)
    if abs(float(hs.double().sum()) - float(gd[name + "_x_sum"])) > 1e-3:
        pytest.skip("torch CPU RNG stream differs from the build that wrote the fixture")
    res = torch.randn(4, 32, 32, 32, generator=torch.manual_seed(1))
    groups, eps, heads = 32, 1e-6, 1           # block defaults: resnet_groups 32, resnet_eps 1e-6, one attention head
    h = hs
    if name in ("UpBlock2D", "CrossAttnUpBlock2D"):
        h = torch.cat([h, res], dim=1)
    h = ounet.resnet_block(sd, "resnets.0", h, temb, groups, eps)
    if "CrossAttn" in name:
        h = ounet.transformer_2d(sd, "attentions.0", h, None, heads, groups, None)   # no text states: attn2 is self-attn
    if name == "UNetMidBlock2DCrossAttn":
        h = ounet.resnet_block(sd, "resnets.1", h, temb, groups, eps)
    elif "Down" in name:
        h = ounet.downsample2d(sd, "downsamplers.0", h)
    else:
        h = ounet.upsample2d(sd, "upsamplers.0", h)
    got = h[0, -1, -3:, -3:].flatten()
    assert torch.allclose(got, torch.tensor(UNET_BLOCK_KNOWN[name]), atol=5e-3), (name, got)


def test_ddim_variance_and_alpha_to_one_constants():
    """schedulers/test_scheduler_ddim.py:94-104 (`_get_variance` constants) and :124-140 (10-step loops with and without
    `set_alpha_to_one`, beta_start = 0.01): the remaining DDIM known answers of the fork's tests."""
    s = osched.OracleDDIM(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear")

    def variance(t, prev_t):       # scheduling_ddim.py:_get_variance
        a_t = s.alphas_cumprod[t]
        a_prev = s.alphas_cumprod[prev_t] if prev_t >= 0 else s.final_alpha_cumprod
        return float(((1 - a_prev) / (1 - a_t)) * (1 - a_t / a_prev))

    for (t, p), want in (((0, 0), 0.0), ((420, 400), 0.14771), ((980, 960), 0.32460), ((487, 486), 0.00979),
                         ((999, 998), 0.02)):
        assert abs(variance(t, p) - want) < 1e-5
    for one, es, em in ((True, 149.8295, 0.1951), (False, 149.0784, 0.1941)):
        s = osched.OracleDDIM(num_train_timesteps=1000, beta_start=0.01, beta_end=0.02, beta_schedule="linear",
                              clip_sample=True, set_alpha_to_one=one)
        s.set_timesteps(10)
        x = _dummy_sample_deter()
        for t in s.timesteps:
            x = s.step(_dummy_model(x, t), t, x)
        assert abs(x.abs().sum().item() - es) < 1e-2
        assert abs(x.abs().mean().item() - em) < 1e-3


def test_tiny_unet_music_golden():
    """The Mustango UNet variant (beat + chord cross-attentions after the text one at every attention position;
    unet_2d_condition_music.py) through the same oracle code path, against the fork's UNet2DConditionModelMusic output
    (tests/golden/tiny_unet_music.npz, oracle/make_golden_music.py) — checker for the "next" row 4."""
    gd = gold("tiny_unet_music.npz")
    cfg = dict(synth.TINY_UNET_CONFIG,
               down_block_types=["CrossAttnDownBlock2DMusic"] * 3 + ["DownBlock2D"],
               mid_block_type="UNetMidBlock2DCrossAttnMusic",
               up_block_types=["UpBlock2D"] + ["CrossAttnUpBlock2DMusic"] * 3)
    sd = {k: synth.synth_tensor(k, eval(shp), 0) for k, shp in zip(gd["keys"].tolist(), gd["shapes"].tolist())}
    assert len(sd) == 1518
    tt = lambda n: torch.from_numpy(gd[n])
    out = ounet.unet_forward(sd, cfg, tt("sample"), torch.tensor(int(gd["t"])), tt("ehs"), tt("mask"),
                             extra_streams=((tt("beat"), tt("bmask")), (tt("chord"), tt("cmask"))))
    assert np.abs(out.numpy() - gd["out"]).max() < 5e-5


def test_config1_artefact_pins_the_oracle_at_full_size():
    """tests/golden/config1.npz (the reference's own config-1 run: full 866 M-parameter UNet, 1 prompt, CFG 3, 10 steps at
    256 x 16, then VAE + HiFi-GAN): the oracle reproduces (a) the first step of both loops — the per-step latent norms the
    reference loop recorded — and (b) mel and int16 waveform from the reference's final DDIM latents. (The full 10-step
    oracle loops are asserted against the reference inside oracle/make_golden_config1.py, ~3 min; here one CFG forward
    per scheduler keeps the CPU suite short.)"""
    from oracle import make_golden_config1 as c1
    gd = np.load(os.path.join(GOLD, "config1.npz"))
    assert gd["timesteps_ddpm"].tolist() == list(range(900, -1, -100))
    assert gd["timesteps_ddim"].tolist() == list(range(901, 0, -100))
    cfg, embeds, mask, lat0, noises = c1.inputs()
    sd = synth.synth_state_dict(synth.unet_param_shapes(cfg), seed=c1.SEEDS["weights"])
    for name, sch in (("ddpm", osched.OracleDDPM(**osched.SD21_CONFIG)), ("ddim", osched.OracleDDIM(**osched.SD21_CONFIG))):
        sch.set_timesteps(c1.STEPS)
        t = sch.timesteps[0]
        x = torch.cat([lat0 * sch.init_noise_sigma] * 2)
        pred = ounet.unet_forward(sd, cfg, x, t, embeds, mask)
        u, c = pred.chunk(2)
        pred = u + c1.GUIDANCE * (c - u)
        lat1 = sch.step(pred, t, lat0, noises[0]) if name == "ddpm" else sch.step(pred, t, lat0)
        want = float(gd[f"step_norms_{name}"][0])
        assert abs(float(lat1.norm()) - want) / want < 2e-6, name
    del sd
    vsd = synth.synth_state_dict(synth.vae_decoder_param_shapes(), seed=c1.SEEDS["weights"])
    lat = torch.from_numpy(gd["latents_ddim"])
    mel = ovae.decode_first_stage(vsd, lat, synth.VAE_CONFIG["scale_factor"])
    _, i16 = ohifi.decode_to_waveform(vsd, mel)
    assert float((mel - torch.from_numpy(gd["mel"])).abs().max()) < 1e-4
    assert int(np.abs(np.asarray(i16).astype(np.int32) - gd["wave_i16"].astype(np.int32)).max()) <= 1
