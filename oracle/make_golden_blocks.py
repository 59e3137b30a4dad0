"""Fixtures for the diffusers fork's own known-answer block tests (TEST INFRASTRUCTURE ONLY; build container only).

mustango/diffusers/tests/test_layers_utils.py builds each block with `torch.manual_seed(0)` default initialisation
and compares an output slice with hard-coded constants. The constants live in tests/test_oracle_pins.py (cited there);
this script reproduces the seeded inputs + module weights through the UNMODIFIED reference modules, checks that the
reference still meets its constants on this torch build, and stores inputs + weights (tests/golden/block_known_answers/,
one file per block) so the oracle's block functions can be checked against the same constants anywhere.

    python -m oracle.make_golden_blocks
"""
import os

import numpy as np
import torch

from oracle import refshim

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

EXPECTED = {   # test_layers_utils.py: ResnetBlock2D :226-240, Upsample2D with conv :131-141, Downsample2D pad 1 :200-210,
               # Transformer2DModel with cross attention :394-418
    "resnet": [-1.9010, -0.2974, -0.8245, -1.3533, 0.8742, -0.9645, -2.0584, 1.3387, -0.4746],
    "upsample": [0.7145, 1.3773, 0.3492, 0.8448, 1.0839, -0.3341, 0.5956, 0.1250, -0.4841],
    "downsample": [0.9267, 0.5878, 0.3337, 1.2321, -0.1191, -0.3984, -0.7532, -0.0715, -0.3913],
    "transformer": [-0.2555, -0.8877, -2.4739, -2.2251, 1.2714, 0.0807, -0.4161, -1.6408, -0.0471],
}


def main():
    torch.set_grad_enabled(False)
    refshim.install()
    from diffusers.models.resnet import Downsample2D, ResnetBlock2D, Upsample2D
    from diffusers.models.transformer_2d import Transformer2DModel
    out = {}

    def check(name, y):
        sl = y[0, -1, -3:, -3:].flatten()
        d = float((sl - torch.tensor(EXPECTED[name])).abs().max())
        print(f"{name}: reference module vs its own hard-coded slice: {d:.2e}")
        assert d < 1e-3

    torch.manual_seed(0)
    x = torch.randn(1, 32, 64, 64)
    temb = torch.randn(1, 128)
    m = ResnetBlock2D(in_channels=32, temb_channels=128)
    check("resnet", m(x, temb))
    out.update({"resnet_x": x, "resnet_temb": temb, **{"resnet." + k: v for k, v in m.state_dict().items()}})

    torch.manual_seed(0)
    x = torch.randn(1, 32, 32, 32)
    m = Upsample2D(channels=32, use_conv=True)
    check("upsample", m(x))
    out.update({"upsample_x": x, **{"upsample." + k: v for k, v in m.state_dict().items()}})

    torch.manual_seed(0)
    x = torch.randn(1, 32, 64, 64)
    m = Downsample2D(channels=32, use_conv=True, padding=1)
    check("downsample", m(x))
    out.update({"downsample_x": x, **{"downsample." + k: v for k, v in m.state_dict().items()}})

    torch.manual_seed(0)
    x = torch.randn(1, 64, 64, 64)
    m = Transformer2DModel(in_channels=64, num_attention_heads=2, attention_head_dim=32, dropout=0.0,
                           cross_attention_dim=64)
    ctx = torch.randn(1, 4, 64)
    check("transformer", m(x, ctx).sample)
    out.update({"transformer_x": x, "transformer_ctx": ctx, **{"transformer." + k: v for k, v in m.state_dict().items()}})

    # the big input tensors are reproducible from the seed (torch CPU RNG): store only a checksum of each
    for k in [k for k in out if k.endswith("_x")]:
        out[k + "_sum"] = out.pop(k).double().sum().float()
    # ---- mustango/diffusers/tests/test_unet_2d_blocks.py + test_unet_blocks_common.py:41-105 (UNetBlockTesterMixin):
    # hidden_states / temb from torch.manual_seed(0), the skip tensor from torch.manual_seed(1), THEN the block is built
    # with default initialisation from the global stream; slices compared at atol 5e-3.
    from diffusers.models import unet_2d_blocks as B

    def common(kind, with_res):
        g = torch.manual_seed(0)
        hs = torch.randn(4, 32, 32, 32, generator=g)
        temb = torch.randn(4, 128, generator=g)
        inp = {"hidden_states": hs, "temb": temb}
        if with_res:
            g1 = torch.manual_seed(1)
            inp["res_hidden_states_tuple"] = (torch.randn(4, 32, 32, 32, generator=g1),)
        init = {"in_channels": 32, "out_channels": 32, "temb_channels": 128}
        if kind == "up":
            init["prev_output_channel"] = 32
        if kind == "mid":
            init.pop("out_channels")
        return init, inp

    UNET_BLOCKS = {   # name: (class, kind, skip input, cross-attention, expected slice (test_unet_2d_blocks.py line))
        "DownBlock2D": (B.DownBlock2D, "down", False, False,
                        [-0.0232, -0.9869, 0.8054, -0.0637, -0.1688, -1.4264, 0.4470, -1.3394, 0.0904]),          # :23-30
        "CrossAttnDownBlock2D": (B.CrossAttnDownBlock2D, "down", False, True,
                                 [0.2440, -0.6953, -0.2140, -0.3874, 0.1966, 1.2077, 0.0441, -0.7718, 0.2800]),    # :50-62
        "UNetMidBlock2DCrossAttn": (B.UNetMidBlock2DCrossAttn, "mid", False, True,
                                    [0.1879, 2.2653, 0.5987, 1.1568, -0.8454, -1.6109, -0.8919, 0.8306, 1.6758]),  # :168-179
        "UpBlock2D": (B.UpBlock2D, "up", True, False,
                      [-0.2041, -0.4165, -0.3022, 0.0041, -0.6628, -0.7053, 0.1928, -0.0325, 0.0523]),            # :200-211
        "CrossAttnUpBlock2D": (B.CrossAttnUpBlock2D, "up", True, True,
                               [-0.2796, -0.4364, -0.1067, -0.2693, 0.1894, 0.3869, -0.3470, 0.4584, 0.5091]),    # :226-241
    }
    for name, (cls, kind, with_res, cross, exp) in UNET_BLOCKS.items():
        init, inp = common(kind, with_res)
        if cross:
            init["cross_attention_dim"] = 32
        blk = cls(**init).eval()
        y = blk(**inp)
        y = y[0] if isinstance(y, tuple) else y
        d = float((y[0, -1, -3:, -3:].flatten() - torch.tensor(exp)).abs().max())
        print(f"{name}: reference block vs its own hard-coded slice: {d:.2e}")
        assert d < 5e-3
        out.update({f"{name}." + k: v for k, v in blk.state_dict().items()})
        out[f"{name}_x_sum"] = inp["hidden_states"].double().sum().float()

    # one file per block (keys keep the block's prefix), so that no fixture file grows past 1 MB
    blocks = sorted(EXPECTED) + sorted(UNET_BLOCKS)
    os.makedirs(os.path.join(GOLD, "block_known_answers"), exist_ok=True)
    for name in blocks:
        part = {k: v.numpy() for k, v in out.items() if k.startswith((name + ".", name + "_"))}
        path = os.path.join(GOLD, "block_known_answers", name + ".npz")
        np.savez_compressed(path, **part)
        print("wrote", path, f"({len(part)} arrays)")
    assert sum(k.startswith((n + ".", n + "_")) for k in out for n in blocks) == len(out)


if __name__ == "__main__":
    main()
