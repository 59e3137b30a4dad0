"""Every launch path of tng_conv_gemm that the workload uses, each pinned to the plan it must reach, checked element by
element against tests/cabi_spec.py:spec_conv_gemm (fp64 on CPU copies of exactly what ops.run_conv hands the kernel);
plus the production-size paths of the GroupNorm-apply, LayerNorm / RMSNorm and cast kernels.

GEMM_CASES is one table: the operator, the epilogue arguments, the plan (block_n, mode, ksplit) the planner must pick
on a 148-SM B200 and where the GroupNorm statistics are computed. If a planner threshold moves, a row fails on its plan
assert and names the plan it got: pick a new shape for that row that reaches the old plan again, so that the row keeps
testing the instantiation it is there for. test_workload_gemm_keys_are_in_the_table runs one CFG UNet step, the VAE
decode and the vocoder at the benchmark shape and fails, naming the key, on any launch path no row covers.

Bounds (per element): fp32 outputs max|got - ref| <= 2e-5 max|ref| (fp32 accumulation of bf16 products); bf16 outputs
|got - ref| <= 2^-8 |ref| + 2e-5 max|ref| (one bf16 rounding of a value that carries the fp32 accumulation error:
near a rounding midpoint that error decides the rounding direction); hi + lo of a split
output within the fp32 bound plus the rounding of lo. Every output is allocated with padding columns and extra rows,
prefilled with NaN (the GroupNorm accumulators with an extra image of a sentinel value), and nothing outside the
written region may change, bit for bit."""
import math
import zlib
from typing import NamedTuple, Optional

import pytest
import torch
import torch.nn.functional as F

import cabi_spec
from tango_b200 import lib as L
from tango_b200 import ops, synth

pytestmark = pytest.mark.gpu

E_F32 = 2e-5
ACT_NAMES = {L.ACT_NONE: "none", L.ACT_SILU: "silu", L.ACT_LRELU: "lrelu", L.ACT_GEGLU: "geglu",
             L.ACT_GEGLU_TANH: "geglu_tanh"}
PAD_ROWS = 5


def gemm_key(plan, f32: bool, bf16: bool, res: Optional[str], split: bool, act: int, stats: Optional[str],
             accumulate: bool) -> str:
    """Launch path of one tng_conv_gemm call: kernel instantiation + epilogue shape."""
    bn, mode, ks = plan
    outs = "+".join(n for n, on in (("f32", f32), ("bf16", bf16)) if on)
    return (f"gemm_tc<{bn},{mode}{',splitk' if ks > 1 else ''}> out={outs} res={res or 'none'} split={int(split)} "
            f"act={ACT_NAMES[act]} stats={stats or 'none'} acc={int(accumulate)}")


def _key_of_call(plan, kw, launches) -> str:
    res = kw.get("res")
    stats = None
    if kw.get("gn_stats") is not None:
        stats = "epilogue" if launches == 1 else "after"
    return gemm_key(plan, kw.get("out_f32") is not None, kw.get("out_bf16") is not None,
                    None if res is None else ("f32" if res.dtype == torch.float32 else "bf16"),
                    kw.get("split_off", 0) > 0, kw.get("act", L.ACT_NONE), stats, bool(kw.get("accumulate", False)))


class Case(NamedTuple):
    name: str
    # operator: kind "conv2d" (k x k, stride), "conv1d" (k taps, dilation) or "linear"; grid NB x H x W (linear: M = W)
    kind: str
    k: int
    Cin: int
    Cout: int
    NB: int
    H: int
    W: int
    plan: tuple                 # (block_n, mode, ksplit) on 148 SMs
    stats: Optional[str] = None  # None, "epilogue" (fused) or "after" (separate pass)
    split: bool = False
    stride: int = 1
    dil: int = 1
    sc: int = 0                 # Cin of a fused 1x1 shortcut (extra k-group)
    geglu: int = 0              # GEGLU N tile (erf GELU)
    bias: bool = True
    rowvec: bool = False
    res: Optional[str] = None   # residual dtype: "f32" / "bf16"
    alpha: float = 1.0
    accumulate: bool = False
    f32: bool = True
    bf16: bool = False
    act: int = L.ACT_NONE
    act_param: float = 0.0
    ld_f32_pad: int = 8         # ld_f32 = Ncols + this (1: misaligned rows -> the scalar epilogue)
    block_n: int = 0

    @property
    def key(self) -> str:
        act = L.ACT_GEGLU if self.geglu else self.act
        return gemm_key(self.plan, self.f32, self.bf16, self.res, self.split and self.bf16, act, self.stats,
                        self.accumulate)


# Plans worked from plan_gemm (tango_b200/csrc/gemm_tc.cu) with 148 SMs. m = M tiles of 128 rows; kit = K blocks of 64
# (x 3 in split mode: hi*hi, lo*hi, hi*lo). Pair mode (4) needs bn 128 / 160, Ncols % (2 bn) == 0, full even M tiling,
# kit >= 36 and (m / 2) * (Ncols / (2 bn)) * 2 >= 74.
GEMM_CASES = [
    # --- <160,4>: 16x16 images in 8-row tiles, m = 40, Ncols 640 -> 20 x 2 pairs; kit = 9 * 4 = 36 (bf16) / 27 * 2 = 54
    Case("pair160_conv1_bf16_rowvec_fused_stats", "conv2d", 3, 256, 640, 20, 16, 16, (160, 4, 1), stats="epilogue",
         rowvec=True, f32=False, bf16=True),
    Case("pair160_conv2_res_alpha_f32_bf16", "conv2d", 3, 256, 640, 20, 16, 16, (160, 4, 1), stats="epilogue",
         res="f32", alpha=0.5, bf16=True, act=L.ACT_SILU),
    Case("pair160_split_hilo", "conv2d", 3, 128, 640, 20, 16, 16, (160, 4, 1), stats="epilogue", split=True,
         rowvec=True, bf16=True, act=L.ACT_SILU),
    # --- <128,4>: VAE-decoder-like 3x3, 128x16 images, m = 16 per image; Ncols 256 (m = 96) / 512 (m = 48): below the
    # 296 N tiles that make 256 the N tile, (m / 2) * (Ncols / 256) * 2 >= 74
    Case("pair128_vae_bf16_res", "conv2d", 3, 256, 256, 6, 128, 16, (128, 4, 1), stats="epilogue", res="f32"),
    Case("pair128_vae_split", "conv2d", 3, 256, 512, 3, 128, 16, (128, 4, 1), stats="epilogue", split=True,
         bf16=True, act=L.ACT_SILU),
    # --- <256,1> chosen by the planner: Ncols 1280 % 256 == 0 and m * 5 = 61 * 5 >= 296; ragged last M tile (20 rows)
    Case("auto256_linear_bf16res_f32_bf16", "linear", 1, 320, 1280, 1, 1, 7700, (256, 1, 1), res="bf16", bf16=True,
         act=L.ACT_LRELU, act_param=0.2),
    # --- <128,1>: Ncols 384 (not % 160, not % 256); split bf16-only hi/lo output, partial last tile
    Case("tile128_linear_split_bf16_only", "linear", 1, 320, 384, 1, 1, 1000, (128, 1, 1), split=True, f32=False,
         bf16=True),
    # --- <160,1,splitk>: 32x2 images (bn = 2 images per tile), 5 images -> m = 3 with a ragged last tile, Ncols 320:
    # 3 * 2 * 2 <= 148 and kit = 90 >= 32 -> two K halves; partial tiles -> statistics in the pass after the GEMM
    Case("splitk160_ragged_rowvec_res", "conv2d", 3, 640, 320, 5, 32, 2, (160, 1, 2), stats="after", rowvec=True,
         res="f32", alpha=0.5),
    # --- <160,1> mode 5 (residual + bf16 only, the UNet feed-forward output): 8 tiles, no split-K with a bf16 output
    Case("tile160_linear_res_bf16_only", "linear", 1, 1280, 320, 1, 1, 1024, (160, 1, 1), res="f32", f32=False,
         bf16=True),
    # --- <32,1> / <64,1>: the vocoder's narrow convolutions
    Case("tile32_conv_post_ncols1", "conv1d", 7, 32, 1, 2, 1, 1000, (32, 1, 1)),
    Case("tile32_conv1d_dilated_bf16_lrelu", "conv1d", 11, 32, 32, 2, 1, 1000, (32, 1, 1), dil=5, f32=False,
         bf16=True, act=L.ACT_LRELU, act_param=0.1),
    Case("tile64_ldf32_odd_scalar_epilogue_res", "conv1d", 3, 64, 64, 2, 1, 700, (64, 1, 1), dil=3, res="f32",
         bf16=True, act=L.ACT_LRELU, act_param=0.1, ld_f32_pad=1),
    Case("tile64_conv1d_dilated_accumulate", "conv1d", 7, 64, 64, 2, 1, 1024, (64, 1, 1), dil=3, res="f32",
         alpha=1.0 / 3, accumulate=True),
    # --- full tiles whose 32-row warp slices span two images (4x4 images, 8 per tile, rpi = 16 < 32) with a row vector
    Case("rpi16_full_tiles_rowvec", "conv2d", 3, 64, 128, 16, 4, 4, (128, 1, 1), stats="after", rowvec=True),
    Case("rpi16_full_tiles_rowvec_res_bf16", "conv2d", 3, 64, 128, 16, 4, 4, (128, 1, 1), rowvec=True, res="bf16",
         f32=False, bf16=True, act=L.ACT_SILU),
    # --- GEGLU (erf) epilogue: split on a partial M tile, and the full-tile bf16 path
    Case("geglu_erf_split_partial_tile", "linear", 1, 128, 512, 1, 1, 300, (256, 1, 1), split=True, geglu=256,
         f32=False, bf16=True),
    Case("geglu_erf_bf16_full_tiles", "linear", 1, 320, 1024, 1, 1, 512, (256, 1, 1), geglu=256, f32=False,
         bf16=True),
    # --- stride-2 (downsample) and a fused 1x1 shortcut k-group
    Case("stride2_down_stats", "conv2d", 3, 128, 128, 4, 32, 32, (128, 1, 1), stats="epilogue", stride=2),
    Case("shortcut_split_f32_stats", "conv2d", 3, 128, 64, 2, 8, 16, (64, 1, 1), stats="epilogue", split=True,
         sc=192),
]


def _vary(base: Case, tag: str, **changes) -> Case:
    return base._replace(name=f"{base.name}__{tag}", **changes)


# The other epilogue shapes the workload launches, on bases whose plan does not depend on the epilogue:
#  <160,4>: 16x16 images, m = 40, Ncols 640 (split: Cin 128, kit 54)
#  <160,1>: linear, m = 8, Ncols 320 (no 128 fallback: 320 % 128 != 0; kit 20 < 32: never split-K; full tiles)
#  <160,1,splitk>: the ragged 32x2 case above
#  <256,1>: linear 7680 rows, m = 60, 60 * 5 >= 296, full tiles
#  <128,1>: stride-2 conv to 16x16, m = 8, kit 18 (split 54 but Ncols 128 is not a multiple of 256: no pair)
#  <32,1> / <64,1>: conv1d over 1024 positions (full tiles)
_P160 = Case("v_pair160", "conv2d", 3, 256, 640, 20, 16, 16, (160, 4, 1))
_P160S = Case("v_pair160_split", "conv2d", 3, 128, 640, 20, 16, 16, (160, 4, 1), split=True)
_T160 = Case("v_tile160", "linear", 1, 1280, 320, 1, 1, 1024, (160, 1, 1))
_T160S = _T160._replace(name="v_tile160_split", Cin=320, split=True)
_SK160 = Case("v_splitk160", "conv2d", 3, 640, 320, 5, 32, 2, (160, 1, 2), rowvec=True)
_T256 = Case("v_tile256", "linear", 1, 320, 1280, 1, 1, 7680, (256, 1, 1))
_T128 = Case("v_tile128", "conv2d", 3, 128, 128, 4, 32, 32, (128, 1, 1), stride=2)
_T32 = Case("v_tile32", "conv1d", 5, 32, 32, 2, 1, 1024, (32, 1, 1), dil=2)
_T64 = Case("v_tile64", "conv1d", 5, 64, 64, 2, 1, 1024, (64, 1, 1), dil=2)
_LRELU = dict(act=L.ACT_LRELU, act_param=0.1)
GEMM_CASES += [
    _vary(_P160, "bf16_res", res="f32", f32=False, bf16=True),
    _vary(_P160S, "bf16_res", res="f32", f32=False, bf16=True),
    _vary(_P160S, "bf16", f32=False, bf16=True),
    _vary(_P160, "res_stats", res="f32", stats="epilogue"),
    _vary(_P160, "res", res="f32"),
    _vary(_P160, "stats", stats="epilogue"),
    _vary(_P160, "plain"),
    _vary(_T160, "bf16", f32=False, bf16=True),
    _vary(_T160S, "bf16", f32=False, bf16=True),
    _vary(_T160S, "bf16_res", res="f32", f32=False, bf16=True),
    _vary(_T160, "res_stats", res="f32", stats="epilogue"),
    _vary(_T160, "res", res="f32"),
    _vary(_T160, "stats", stats="epilogue"),
    _vary(_T160, "plain"),
    _vary(_SK160, "stats", stats="after"),
    _vary(_SK160, "plain"),
    _vary(_T256, "bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T256._replace(split=True), "split_bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T256, "bf16", f32=False, bf16=True),
    _vary(_T256._replace(split=True), "split_bf16", f32=False, bf16=True),
    _vary(_T256, "res_stats", res="f32", stats="epilogue"),
    _vary(_T256, "res", res="f32"),
    _vary(_T256, "res_acc", res="f32", accumulate=True, alpha=0.25),
    _vary(_T256, "stats", stats="epilogue"),
    _vary(_T256, "plain"),
    _vary(_T256, "res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T256._replace(split=True), "split_res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T128, "bf16_res", res="f32", f32=False, bf16=True),
    _vary(_T128._replace(split=True), "split_bf16_res", res="f32", f32=False, bf16=True),
    _vary(_T128, "bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T128._replace(split=True), "split_bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T128, "bf16", f32=False, bf16=True),
    _vary(_T128._replace(split=True), "split_bf16", f32=False, bf16=True),
    _vary(_T128, "res_stats", res="f32", stats="epilogue"),
    _vary(_T128, "res", res="f32"),
    _vary(_T128, "res_acc", res="f32", accumulate=True, alpha=0.25),
    _vary(_T128, "plain"),
    _vary(_T128, "res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T128._replace(split=True), "split_res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T32._replace(split=True), "split_bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T32, "res", res="f32"),
    _vary(_T32, "res_acc", res="f32", accumulate=True, alpha=0.25),
    _vary(_T32, "res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T32._replace(split=True), "split_res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T64, "bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T64._replace(split=True), "split_bf16_lrelu", f32=False, bf16=True, **_LRELU),
    _vary(_T64, "res", res="f32"),
    _vary(_T64, "res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
    _vary(_T64._replace(split=True), "split_res_f32_bf16_lrelu", res="f32", bf16=True, **_LRELU),
]


def _host(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """CPU copy with the same layout (a view keeps its strides and offset into a copy of its base)."""
    if t is None:
        return None
    base = t if t._base is None else t._base
    hb = base.detach().cpu()
    return hb.as_strided(t.shape, t.stride(), t.storage_offset() - base.storage_offset())


class _Recorder:
    """Stands in for lib.conv_gemm: records the plan, the launch count and (optionally) CPU copies of the operands."""

    def __init__(self, real, snapshot: bool):
        self.real, self.snapshot, self.calls = real, snapshot, []

    def __call__(self, views, groups, weight, W, H, NB, **kw):
        rec = {"plan": L.gemm_plan(views, groups, weight, W, H, NB, **kw)}
        if self.snapshot:
            torch.cuda.synchronize()
            rec["views"] = [L.View(_host(v.t), v.C, v.W, v.H, v.NB, v.s_w, v.s_h, v.s_n, v.off) for v in views]
            rec["groups"], rec["weight"], rec["grid"] = list(groups), weight.cpu(), (W, H, NB)
            rec["kw"] = {k: (_host(v) if isinstance(v, torch.Tensor) else v) for k, v in kw.items()}
        n0 = L.launch_count()
        self.real(views, groups, weight, W, H, NB, **kw)
        rec["launches"] = L.launch_count() - n0
        rec["key"] = _key_of_call(rec["plan"], kw, rec["launches"])
        self.calls.append(rec)


def _bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float64: torch.int64}[t.dtype])


def _assert_outside_unchanged(before, after, keep, what):
    changed = (_bits(before) != _bits(after)) & ~keep
    assert not changed.any(), f"{what}: {int(changed.sum())} elements written outside the output region, first at " \
                              f"{changed.nonzero()[0].tolist()}"


def _bf16_bound(got, z, what):
    err = (got.double() - z.double()).abs()
    lim = 2.0 ** -8 * z.double().abs() + E_F32 * z.double().abs().max()
    bad = ~(err <= lim)
    assert not bad.any(), f"{what}: {int(bad.sum())} elements beyond one bf16 rounding, worst at " \
                          f"{(err - lim).argmax().item()}"


def _f32_bound(got, ref, what, extra=None):
    err = (got.double() - ref.double()).abs()
    lim = E_F32 * ref.double().abs().max() + (0 if extra is None else extra)
    bad = ~(err <= lim)
    assert not bad.any(), f"{what}: {int(bad.sum())} elements beyond the fp32 bound, max err " \
                          f"{err.max().item():.3e} vs {float(lim if extra is None else lim.max()):.3e}"


def _build(case: Case, dev):
    """Packed layer, bf16 input rows (hi | lo in split mode), run_conv keywords and the fp32 source tensors."""
    g = torch.Generator(device="cpu").manual_seed(zlib.crc32(case.name.encode()))
    NB, H, W, Cin, Cout = case.NB, case.H, case.W, case.Cin, case.Cout
    if case.kind == "conv2d":
        x = torch.randn(NB, Cin, H, W, generator=g)
        w = torch.randn(Cout, Cin, case.k, case.k, generator=g) / math.sqrt(case.k * case.k * Cin)
        rows_in = x.permute(0, 2, 3, 1).reshape(-1, Cin)
    elif case.kind == "conv1d":
        x = torch.randn(NB, Cin, W, generator=g)
        w = torch.randn(Cout, Cin, case.k, generator=g) / math.sqrt(case.k * Cin)
        rows_in = x.permute(0, 2, 1).reshape(-1, Cin)
    else:
        x = torch.randn(W, Cin, generator=g)
        w = torch.randn(Cout, Cin, generator=g) / math.sqrt(Cin)
        rows_in = x
    b = torch.randn(Cout, generator=g) if case.bias else None
    sc_w = sc_x = sc_rows = None
    if case.sc:
        sc_x = torch.randn(NB, case.sc, H, W, generator=g)
        sc_w = torch.randn(Cout, case.sc, 1, 1, generator=g) / math.sqrt(case.sc)
        sc_rows = sc_x.permute(0, 2, 3, 1).reshape(-1, case.sc)
    pc = ops.PackedConv(w.to(dev), None if b is None else b.to(dev), split=case.split, device=dev, stride=case.stride,
                        dilation=case.dil, geglu_bn=case.geglu, sc_w=None if sc_w is None else sc_w.to(dev))

    def operand(r):
        r = r.contiguous()
        if not case.split:
            return r.to(torch.bfloat16).to(dev)
        hi = r.to(torch.bfloat16)
        return torch.cat([hi, (r - hi.float()).to(torch.bfloat16)], dim=1).contiguous().to(dev)

    Ho, Wo = (H + case.stride - 1) // case.stride, (W + case.stride - 1) // case.stride
    rows, Nz = NB * Ho * Wo, (Cout // 2 if case.geglu else Cout)
    kw = {}
    if case.rowvec:
        kw["rowvec"] = torch.randn(NB, Cout, generator=g).to(dev)
    if case.res:
        r = torch.randn(rows, Cout, generator=g)
        kw["res"] = (r if case.res == "f32" else r.to(torch.bfloat16)).to(dev)
    if case.alpha != 1.0:
        kw["alpha"] = case.alpha
    if case.act != L.ACT_NONE:
        kw["act"], kw["act_param"] = case.act, case.act_param
    src = dict(x=x, w=w, b=b, sc_x=sc_x, sc_w=sc_w, rows=rows, Nz=Nz, Ho=Ho, Wo=Wo)
    return pc, operand(rows_in), (operand(sc_rows) if case.sc else None), kw, src


def _torch_fp64(case: Case, src, kw, dev):
    """fp64 torch evaluation of the layer on the UNROUNDED fp32 operands (split rows: ~fp32 accuracy expected)."""
    x, w, b = src["x"].double().to(dev), src["w"].double().to(dev), src["b"]
    bd = None if b is None else b.double().to(dev)
    if case.kind == "conv2d":
        y = F.conv2d(x, w, bd, stride=case.stride, padding=case.k // 2)
        if case.sc:
            y = y + F.conv2d(src["sc_x"].double().to(dev), src["sc_w"].double().to(dev))
        y = y.permute(0, 2, 3, 1).reshape(src["rows"], -1)
    elif case.kind == "conv1d":
        y = F.conv1d(x, w, bd, padding=(case.k * case.dil - case.dil) // 2, dilation=case.dil)
        y = y.permute(0, 2, 1).reshape(src["rows"], -1)
    else:
        y = F.linear(x, w, bd)
    if case.rowvec:
        y = y + kw["rowvec"].double().repeat_interleave(src["Ho"] * src["Wo"], 0)
    if case.res:
        y = y + kw["res"].double()
    y = y * case.alpha
    if case.geglu:
        inner = case.Cout // 2
        return y, y[:, :inner] * F.gelu(y[:, inner:])
    z = F.silu(y) if case.act == L.ACT_SILU else F.leaky_relu(y, case.act_param) if case.act == L.ACT_LRELU else y
    return y, z


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c.name for c in GEMM_CASES])
def test_gemm_launch_path(cuda, monkeypatch, case: Case):
    pc, xin, scin, kw, src = _build(case, cuda)
    rows, N, Nz = src["rows"], case.Cout, src["Nz"]
    nan = float("nan")
    bufs = {}
    if case.f32:
        bufs["f32"] = torch.full((rows + PAD_ROWS, N + case.ld_f32_pad), nan, device=cuda)
        if case.accumulate:
            bufs["f32"][:rows, :N] = torch.randn(rows, N, device=cuda)
        kw["out_f32"] = bufs["f32"][:rows, :N]
    wb = Nz * (2 if case.split else 1)
    if case.bf16:
        bufs["bf16"] = torch.full((rows + PAD_ROWS, wb + 8), nan, device=cuda, dtype=torch.bfloat16)
        kw["out_bf16"] = bufs["bf16"][:rows, :wb]
    nimg = case.NB
    if case.stats:
        bufs["stats"] = torch.zeros(nimg + 1, N, 2, device=cuda, dtype=torch.float64)
        bufs["stats"][nimg] = 12345.0
        kw["gn_stats"], kw["stats_hw"] = bufs["stats"][:nimg], src["Ho"] * src["Wo"]
    before = {k: v.clone() for k, v in bufs.items()}

    rec = _Recorder(L.conv_gemm, snapshot=True)
    monkeypatch.setattr(L, "conv_gemm", rec)
    ops.run_conv(pc, xin, case.NB, case.H, case.W, sc_x=scin, accumulate=case.accumulate, block_n=case.block_n, **kw)
    torch.cuda.synchronize()
    assert len(rec.calls) == 1
    call = rec.calls[0]
    assert tuple(call["plan"]) == case.plan, \
        f"the planner now picks {call['plan']} for this row, which is there to test {case.plan}: choose a new shape " \
        f"that reaches {case.plan}"
    assert call["launches"] == (2 if case.stats == "after" else 1), \
        f"{call['launches']} launches: statistics expected {'after the GEMM' if case.stats == 'after' else 'fused'}"
    assert call["key"] == case.key

    # fp64 reference of the same descriptor on CPU copies of the operands. Its fp32 epilogue value y always goes to an
    # fp32 buffer (a scratch one when the row has no fp32 output); the bf16 output is checked against z = act(y),
    # unrounded, so that one bf16 rounding is all the bound has to allow.
    hkw = dict(call["kw"])
    so = hkw.get("split_off", 0)
    assert so == (Nz if (case.split and case.bf16) else 0)
    if not case.f32:
        hkw["out_f32"] = torch.zeros(rows, N)
    hkw["out_bf16"] = None
    if case.stats:
        hkw["gn_stats"] = torch.zeros(nimg, N, 2, dtype=torch.float64)
    W_, H_, NB_ = call["grid"]
    cabi_spec.spec_conv_gemm(call["views"], call["groups"], call["weight"], W_, H_, NB_, **hkw)
    y = hkw["out_f32"][:, :N].double()

    if case.f32:
        got = bufs["f32"][:rows, :N].cpu()
        _f32_bound(got, y, "fp32 output")
        keep = torch.zeros_like(bufs["f32"], dtype=torch.bool)
        keep[:rows, :N] = True
        _assert_outside_unchanged(before["f32"], bufs["f32"], keep, "fp32 output")
    if case.bf16:
        if case.geglu:
            t = y.view(rows, N // case.geglu, case.geglu)
            z = (t[..., :case.geglu // 2] * F.gelu(t[..., case.geglu // 2:])).reshape(rows, Nz)
        else:
            z = F.silu(y) if case.act == L.ACT_SILU else F.leaky_relu(y, case.act_param) if case.act == L.ACT_LRELU else y
        hi = bufs["bf16"][:rows, :Nz].cpu()
        _bf16_bound(hi, z, "bf16 output")
        keep = torch.zeros_like(bufs["bf16"], dtype=torch.bool)
        keep[:rows, :Nz] = True
        if case.split:
            rec_z = hi.float() + bufs["bf16"][:rows, Nz:2 * Nz].cpu().float()
            _f32_bound(rec_z, z, "hi + lo output", extra=2.0 ** -16 * z.double().abs())
            keep[:rows, Nz:2 * Nz] = True
        _assert_outside_unchanged(before["bf16"], bufs["bf16"], keep, "bf16 output")
    if case.stats:
        st = bufs["stats"][:nimg].cpu()
        hw = src["Ho"] * src["Wo"]
        if case.f32 or case.stats == "after":
            # the sums of what was stored (fp32 output, else the bf16 output the pass after the GEMM reads)
            o = (bufs["f32"][:rows, :N] if case.f32 else bufs["bf16"][:rows, :N]).cpu().double().view(nimg, hw, N)
            s_ref, q_ref, e = o.sum(1), (o * o).sum(1), 0.0
            a_sum = o.abs().sum(1)
        else:
            # fused statistics of a bf16-only output: sums of the fp32 epilogue values, which are not stored; each lies
            # within e of the reference value
            s_ref, q_ref = hkw["gn_stats"][..., 0], hkw["gn_stats"][..., 1]
            a_sum = y.view(nimg, hw, N).abs().sum(1)
            e = E_F32 * y.abs().max().item()
        assert ((st[..., 0] - s_ref).abs() <= 1e-6 * a_sum + hw * e).all(), "GroupNorm sums"
        assert ((st[..., 1] - q_ref).abs() <= 1e-6 * q_ref + 2 * e * a_sum + hw * e * e).all(), "GroupNorm sums of squares"
        keep = torch.zeros_like(bufs["stats"], dtype=torch.bool)
        keep[:nimg] = True
        _assert_outside_unchanged(before["stats"], bufs["stats"], keep, "GroupNorm accumulators")

    if case.split:
        y, zt = _torch_fp64(case, src, kw, cuda)
        if case.f32:
            assert cabi_rel(bufs["f32"][:rows, :N], y) < 3e-5
        if case.bf16:
            got = bufs["bf16"][:rows, :Nz].float() + bufs["bf16"][:rows, Nz:2 * Nz].float()
            assert cabi_rel(got, zt) < 3e-5


def cabi_rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


# ------------------------------------------------------------------------------------ coverage of the workload's GEMMs
@pytest.mark.parametrize("precision", ["bf16", "split"])
def test_workload_gemm_keys_are_in_the_table(cuda, monkeypatch, precision):
    """One CFG UNet step at the benchmark shape (8 prompts -> UNet batch 16, 256 x 16 latents, 64 tokens), then the
    VAE decoder and the vocoder for those 8 latents, eagerly: every launch path they take must be a row of GEMM_CASES."""
    from tango_b200.pipeline import Tango

    torch.set_grad_enabled(False)
    cfg = synth.BASE_UNET_CONFIG
    t = Tango.from_synthetic(unet_config=cfg, device=cuda, precision=precision)
    t.model.use_cuda_graph = False
    B = 8
    embeds, mask = synth.synth_conditioning(B, 64, cfg["cross_attention_dim"], seed=1)
    rec = _Recorder(L.conv_gemm, snapshot=False)
    monkeypatch.setattr(L, "conv_gemm", rec)
    gen = torch.Generator(device=cuda).manual_seed(1234)
    lat = t.model.inference([f"p{i}" for i in range(B)], t.scheduler, 1, 3.0, prompt_embeds=embeds.to(cuda),
                            boolean_prompt_mask=mask.to(cuda), generator=gen, latent_shape=(256, 16))
    Bl, Cl, H, W = lat.shape
    rows = lat.permute(0, 2, 3, 1).reshape(Bl * H * W, Cl).contiguous()
    t.vae.decode_rows_to_waveform(rows, Bl, H, W, use_cuda_graph=False)
    torch.cuda.synchronize()
    seen = {}
    for c in rec.calls:
        seen[c["key"]] = seen.get(c["key"], 0) + 1
    print(f"\n[{precision}] {len(rec.calls)} tng_conv_gemm launches, {len(seen)} launch paths:")
    for k in sorted(seen):
        print(f"  {seen[k]:5d}  {k}")
    table = {c.key for c in GEMM_CASES}
    missing = sorted(k for k in seen if k not in table)
    assert not missing, "launch paths of the workload that no row of GEMM_CASES tests:\n  " + "\n  ".join(missing)


# ------------------------------------------------------------------------------- production-size elementwise kernels
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("NB,HW,C0,C1,dt1", [(16, 4096, 320, 0, None), (16, 1024, 640, 320, torch.bfloat16)])
def test_groupnorm_apply_production_size(cuda, NB, HW, C0, C1, dt1):
    """gn_apply at the UNet's level-1 size (fp32 in, SiLU, hi | lo output and raw copy) and the 640 + 320 skip concat.
    A CTA of 256 threads covers one channel slab with RL = 256 // (slab / 4) row lanes; at most 8 such CTAs are
    resident per SM, so the one-wave grid has at most 8 * SMs / (NB * slabs) pixel blocks per (image, slab) and each
    thread walks more than 8 rows: the rows are loaded in several batches of <= 8 (the balanced `per`), not one."""
    C = C0 + C1
    cpg = C // 32
    gps = 1
    while (gps * cpg) % 4:
        gps += 1
    while gps * 2 * cpg <= 320 and 32 % (gps * 2) == 0:
        gps *= 2
    slab = gps * cpg
    RL = 256 // min(slab // 4, 256)
    blocks = max(1, 8 * _sms() // (NB * (32 // gps)))
    min_rows_per_thread = math.ceil(HW / blocks) // RL
    assert min_rows_per_thread > 8, min_rows_per_thread

    g = torch.Generator(device="cpu").manual_seed(HW + C)
    x0 = (torch.randn(NB * HW, C0, generator=g) * 2 + 0.5).to(cuda)
    x1 = torch.randn(NB * HW, C1, generator=g).to(dt1).to(cuda) if C1 else None
    gamma = torch.randn(C, generator=g).to(cuda)
    beta = torch.randn(C, generator=g).to(cuda)
    st0 = torch.zeros(NB, C0, 2, device=cuda, dtype=torch.float64)
    L.groupnorm_stats(x0, NB, HW, st0)
    st1 = None
    if C1:
        st1 = torch.zeros(NB, C1, 2, device=cuda, dtype=torch.float64)
        L.groupnorm_stats(x1, NB, HW, st1)
    rows = NB * HW
    ybuf = torch.full((rows + PAD_ROWS, 2 * C + 8), float("nan"), device=cuda, dtype=torch.bfloat16)
    rbuf = torch.full((rows + PAD_ROWS, 2 * C + 8), float("nan"), device=cuda, dtype=torch.bfloat16)
    y0, r0 = ybuf.clone(), rbuf.clone()
    L.groupnorm(x0, st0, x1, st1, NB, HW, 32, gamma, beta, 1e-5, L.ACT_SILU, ybuf[:rows, :2 * C], split_off=C,
                raw=rbuf[:rows, :2 * C], raw_split_off=C)
    xc = x0.double() if x1 is None else torch.cat([x0.double(), x1.double()], dim=1)
    ref = F.group_norm(xc.view(NB, HW, C).permute(0, 2, 1), 32, gamma.double(), beta.double(), 1e-5)
    ref = F.silu(ref).permute(0, 2, 1).reshape(rows, C)
    torch.cuda.synchronize()
    got = ybuf[:rows, :C].double() + ybuf[:rows, C:2 * C].double()
    # fp32 normalisation (statistics from fp64 sums): ~1e-6 of the output scale per element
    assert ((got - ref).abs() <= 2e-5 * ref.abs().max()).all()
    _bf16_bound(ybuf[:rows, :C].cpu(), ref.cpu(), "GroupNorm hi")
    raw_got = rbuf[:rows, :C].double() + rbuf[:rows, C:2 * C].double()
    assert ((raw_got - xc).abs() <= 2.0 ** -16 * xc.abs()).all()
    keep = torch.zeros_like(ybuf, dtype=torch.bool)
    keep[:rows, :2 * C] = True
    _assert_outside_unchanged(y0, ybuf, keep, "GroupNorm output")
    _assert_outside_unchanged(r0, rbuf, keep, "GroupNorm raw copy")


@pytest.mark.parametrize("rms", [False, True])
@pytest.mark.parametrize("Cc", [64, 256, 320, 640, 1280, 2048])
def test_layernorm_stride_loop(cuda, Cc, rms):
    """rows = 3 * (4 * SMs CTAs * 8 warps) + 5: the grid is capped at 4 CTAs of 8 warps per SM, so every warp walks 3 or
    4 rows (row stride loop + next-row prefetch) and the last 5 rows are a ragged tail. C = 64 ... 2048 selects
    NI = 1, 2, 3, 5, 10 and 16 float4 per lane."""
    rows = 3 * 4 * _sms() * 8 + 5
    g = torch.Generator(device="cpu").manual_seed(Cc + rms)
    x = (torch.randn(rows, Cc, generator=g) * 3 + 1).to(cuda)
    gamma = torch.randn(Cc, generator=g).to(cuda)
    beta = torch.randn(Cc, generator=g).to(cuda)
    ybuf = torch.full((rows + PAD_ROWS, 2 * Cc + 8), float("nan"), device=cuda, dtype=torch.bfloat16)
    y0 = ybuf.clone()
    xd = x.double()
    if rms:
        yf = torch.full((rows, Cc), float("nan"), device=cuda)
        L.rmsnorm(x, gamma, 1e-6, ybuf[:rows, :2 * Cc], split_off=Cc, y_f32=yf)
        ref = gamma.double() * xd * torch.rsqrt(xd.pow(2).mean(-1, keepdim=True) + 1e-6)
    else:
        L.layernorm(x, gamma, beta, 1e-5, ybuf[:rows, :2 * Cc], split_off=Cc)
        ref = F.layer_norm(xd, (Cc,), gamma.double(), beta.double(), 1e-5)
    torch.cuda.synchronize()
    lim = 1e-5 * ref.abs().max()
    got = ybuf[:rows, :Cc].double() + ybuf[:rows, Cc:2 * Cc].double()
    assert ((got - ref).abs() <= lim).all()
    _bf16_bound(ybuf[:rows, :Cc].cpu(), ref.cpu(), "norm hi")
    if rms:
        assert ((yf.double() - ref).abs() <= lim).all()
    keep = torch.zeros_like(ybuf, dtype=torch.bool)
    keep[:rows, :2 * Cc] = True
    _assert_outside_unchanged(y0, ybuf, keep, "norm output")


@pytest.mark.parametrize("up,act,split", [(False, L.ACT_NONE, False), (True, L.ACT_LRELU, False),
                                          (False, L.ACT_SILU, True), (True, L.ACT_NONE, True)])
def test_cast_act_batched_grid(cuda, up, act, split):
    """cast_act's grid is capped at 16 * SMs CTAs of 256 threads and each thread issues the loads of 4 grid-stride
    iterations before its stores: more than 4 * 16 * SMs * 256 output quads (plus a tail) run a second batch and a
    partial one. NONE / LRELU outputs are exactly torch's bf16 rounding; SiLU within one bf16 ulp."""
    C = 320
    Q = C // 4
    stride_quads = 16 * _sms() * 256
    out_quads = 4 * stride_quads + stride_quads // 2 + 3 * Q     # + a partial batch; whole rows
    out_rows = -(-out_quads // Q)
    NB, W = 1, 16
    if up:
        H = -(-out_rows // (4 * W))
        out_rows = 4 * NB * H * W
    else:
        H = -(-out_rows // W)
        out_rows = NB * H * W
    assert out_rows * Q > 4 * stride_quads
    g = torch.Generator(device="cpu").manual_seed(out_rows + act)
    in_rows = NB * H * W
    xbuf = (torch.randn(in_rows, C + 4, generator=g) * 3).to(cuda)    # ld_x = C + 4
    x = xbuf[:, :C]
    wy = 2 * C if split else C
    ybuf = torch.full((out_rows + PAD_ROWS, wy + 8), float("nan"), device=cuda, dtype=torch.bfloat16)
    y0 = ybuf.clone()
    L.cast_act(x, NB, H, W, ybuf[:out_rows, :wy], Cc=C, upsample2x=up, act=act, act_param=0.1,
               split_off=C if split else 0)
    # NONE / LRELU: the fp32 value (x * 0.1f, one rounding, as torch's fp32 leaky_relu) rounded once to bf16
    zf = F.leaky_relu(x, 0.1) if act == L.ACT_LRELU else x.clone()
    z = F.silu(x.double()) if act == L.ACT_SILU else zf.double()
    if up:
        z = z.view(NB, H, W, C).repeat_interleave(2, 1).repeat_interleave(2, 2).reshape(out_rows, C)
        zf = zf.view(NB, H, W, C).repeat_interleave(2, 1).repeat_interleave(2, 2).reshape(out_rows, C)
    torch.cuda.synchronize()
    hi = ybuf[:out_rows, :C]
    if act == L.ACT_SILU:
        ulp = torch.finfo(torch.bfloat16).eps * z.abs()         # >= one bf16 ulp of the value
        assert ((hi.double() - z).abs() <= ulp).all()
    else:
        assert torch.equal(hi, zf.to(torch.bfloat16))
    if split:
        # lo = bf16(z - hi): off by at most 2^-8 |z - hi| <= 2^-16 |z| (+ the fp32 SiLU)
        rec = hi.double() + ybuf[:out_rows, C:2 * C].double()
        assert ((rec - z).abs() <= 2.0 ** -16 * z.abs() + 1e-6 * z.abs().max()).all()
    keep = torch.zeros_like(ybuf, dtype=torch.bool)
    keep[:out_rows, :wy] = True
    _assert_outside_unchanged(y0, ybuf, keep, "cast output")
