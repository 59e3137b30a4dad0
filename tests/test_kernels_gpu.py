"""Per-kernel numerics on the GPU: each hand-written kernel against a plain PyTorch fp32 evaluation of the same op
on the same (bf16-rounded) operands. Model-level parity against the oracle lives in test_parity_gpu.py."""
import math

import pytest
import torch
import torch.nn.functional as F

from tango_b200 import lib as L
from tango_b200 import ops
from tango_b200.ops import PackedConv, run_conv

pytestmark = pytest.mark.gpu


def bf(x):
    return x.to(torch.bfloat16)


def rel_err(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12)).item()


def run_conv_planned(monkeypatch, *args, **kw):
    """ops.run_conv, returning ((block_n, mode, ksplit), launches) of the one tng_conv_gemm call it makes: the plan
    lib.gemm_plan reports for that descriptor, and 1 launch (statistics in the epilogue) or 2 (pass after the GEMM)."""
    real, seen = L.conv_gemm, []

    def rec(views, groups, weight, W, H, NB, **k):
        plan = L.gemm_plan(views, groups, weight, W, H, NB, **k)
        n0 = L.launch_count()
        real(views, groups, weight, W, H, NB, **k)
        seen.append((plan, L.launch_count() - n0))

    with monkeypatch.context() as m:
        m.setattr(L, "conv_gemm", rec)
        ops.run_conv(*args, **kw)
    assert len(seen) == 1
    return seen[0]


def nhwc_rows(x):  # [N,C,H,W] -> [N*H*W, C]
    return x.permute(0, 2, 3, 1).reshape(-1, x.shape[1]).contiguous()


def to_split(x_f32):  # [rows, C] fp32 -> bf16 [rows, 2C] = [hi | lo]
    hi = bf(x_f32)
    lo = bf(x_f32 - hi.float())
    return torch.cat([hi, lo], dim=1).contiguous()


@pytest.mark.parametrize("M,K,N,bn", [(300, 192, 320, 0), (128, 64, 256, 256), (1000, 320, 128, 128),
                                      (77, 128, 64, 64), (513, 256, 8, 0), (4096, 1280, 1280, 0)])
def test_linear(cuda, M, K, N, bn):
    g = torch.Generator(device="cpu").manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g).to(cuda)
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(cuda)
    b = torch.randn(N, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=False, device=cuda)
    xb = bf(x)
    of = torch.full((M, N), float("nan"), device=cuda)
    ob = torch.zeros(M, N, device=cuda, dtype=torch.bfloat16)
    ops.run_linear(pc, xb, out_f32=of, out_bf16=ob, block_n=bn)
    ref = xb.float() @ bf(w).float().t() + b
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 2e-5
    assert rel_err(ob, ref) < 5e-3


@pytest.mark.parametrize("NB,H,W,Cin,Cout", [(2, 32, 16, 64, 128), (3, 8, 4, 128, 320), (2, 4, 2, 192, 64),
                                             (1, 16, 64, 64, 32), (2, 12, 16, 8, 64), (1, 64, 16, 320, 8)])
def test_conv3x3(cuda, NB, H, W, Cin, Cout):
    g = torch.Generator(device="cpu").manual_seed(NB * 1000 + H + Cin)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    temb = torch.randn(NB, Cout, generator=g).to(cuda)
    res = torch.randn(NB * H * W, Cout, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=False, device=cuda)
    xb = bf(nhwc_rows(x))
    of = torch.full((NB * H * W, Cout), float("nan"), device=cuda)
    ops.run_conv(pc, xb, NB, H, W, rowvec=temb, res=res, alpha=0.5, out_f32=of)
    ref = F.conv2d(bf(x).float(), bf(w).float(), b, padding=1) + temb[:, :, None, None]
    ref = (nhwc_rows(ref) + res) * 0.5
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 2e-5


# Pair mode needs >= 36 K blocks of 64 (9 taps x Cin / 64, x 3 in split mode) and (pairs) x (N pairs) x 2 >= SMs / 2
@pytest.mark.parametrize("NB,H,W,Cin,Cout,split", [(5, 32, 64, 256, 320, False),     # 40 pair tiles x 1 N pair
                                                   (20, 16, 16, 256, 640, False),    # 20 x 2, W < 128 pixel tiles
                                                   (20, 8, 64, 128, 256, True),      # N tile 128 x 2, hi/lo K groups
                                                   (4, 64, 16, 320, 1280, False)])   # 16 x 4, the UNet level-2 shape
def test_conv3x3_pair_tiles_two_accumulators(cuda, monkeypatch, NB, H, W, Cin, Cout, split):
    """Launches large enough for the CTA-pair mode (tcgen05 cta_group::2, 256 x 2*BN output tile per pair, two
    accumulators in a 3-slot TMEM ring): full epilogue with bias, time-embedding row vector, residual, fp32 + bf16
    (SiLU) outputs and the GroupNorm statistics, against torch."""
    g = torch.Generator(device="cpu").manual_seed(NB * 100 + Cout)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    temb = torch.randn(NB, Cout, generator=g).to(cuda)
    res = torch.randn(NB * H * W, Cout, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=split, device=cuda)
    rows = nhwc_rows(x)
    xin = to_split(rows) if split else bf(rows)
    of = torch.full((NB * H * W, Cout), float("nan"), device=cuda)
    ob = torch.zeros(NB * H * W, Cout * (2 if split else 1), device=cuda, dtype=torch.bfloat16)
    st = torch.zeros(NB, Cout, 2, device=cuda, dtype=torch.float64)
    plan, launches = run_conv_planned(monkeypatch, pc, xin, NB, H, W, rowvec=temb, res=res, out_f32=of, out_bf16=ob,
                                      act=L.ACT_SILU, gn_stats=st, stats_hw=H * W)
    assert plan == ((128, 4, 1) if split else (160, 4, 1)), f"{plan}: choose a shape that reaches the pair mode again"
    assert launches == 1      # statistics from the epilogue
    if split:
        ref = F.conv2d(x.double(), w.double(), b.double(), padding=1).float()
    else:
        ref = F.conv2d(bf(x).float(), bf(w).float(), b, padding=1)
    ref = nhwc_rows(ref + temb[:, :, None, None]) + res
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 3e-5
    got_b = ob[:, :Cout].float() + (ob[:, Cout:].float() if split else 0)
    assert rel_err(got_b, F.silu(ref)) < (3e-5 if split else 5e-3)
    o = of.double().view(NB, H * W, Cout)
    assert rel_err(st[..., 0], o.sum(1)) < 1e-6 and rel_err(st[..., 1], (o * o).sum(1)) < 1e-6


def test_conv3x3_split_matches_fp32(cuda):
    NB, H, W, Cin, Cout = 2, 16, 16, 128, 160
    g = torch.Generator(device="cpu").manual_seed(5)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=True, device=cuda)
    xs = to_split(nhwc_rows(x))
    of = torch.empty(NB * H * W, Cout, device=cuda)
    ob = torch.empty(NB * H * W, 2 * Cout, device=cuda, dtype=torch.bfloat16)
    ops.run_conv(pc, xs, NB, H, W, out_f32=of, out_bf16=ob, act=L.ACT_SILU)
    ref = nhwc_rows(F.conv2d(x.double(), w.double(), b.double(), padding=1)).float()
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 3e-5
    act = F.silu(ref)
    rec = ob[:, :Cout].float() + ob[:, Cout:].float()
    assert rel_err(rec, act) < 3e-5


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("Cin", [8, 64])
def test_conv3x3_small_cin_split_views(cuda, split, Cin):
    NB, H, W, Cout = 2, 8, 16, 64
    g = torch.Generator(device="cpu").manual_seed(11)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    pc = ops.PackedConv(w, None, split=split, device=cuda)
    rows = nhwc_rows(x)
    xin = to_split(rows) if split else bf(rows)
    of = torch.empty(NB * H * W, Cout, device=cuda)
    ops.run_conv(pc, xin, NB, H, W, out_f32=of)
    if split:
        ref = nhwc_rows(F.conv2d(x.double(), w.double(), padding=1)).float()
        tol = 3e-5
    else:
        ref = nhwc_rows(F.conv2d(bf(x).float(), bf(w).float(), padding=1))
        tol = 2e-5
    torch.cuda.synchronize()
    assert rel_err(of, ref) < tol


@pytest.mark.parametrize("split", [False, True])
def test_conv_stride2(cuda, split):
    NB, H, W, Cin, Cout = 2, 16, 8, 64, 128
    g = torch.Generator(device="cpu").manual_seed(7)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=split, device=cuda, stride=2)
    rows = nhwc_rows(x)
    xin = to_split(rows) if split else bf(rows)
    of = torch.empty(NB * (H // 2) * (W // 2), Cout, device=cuda)
    ops.run_conv(pc, xin, NB, H, W, out_f32=of)
    if split:
        ref = F.conv2d(x.double(), w.double(), b.double(), stride=2, padding=1).float()
    else:
        ref = F.conv2d(bf(x).float(), bf(w).float(), b, stride=2, padding=1)
    torch.cuda.synchronize()
    assert rel_err(of, nhwc_rows(ref)) < 3e-5


@pytest.mark.parametrize("split", [False, True])
def test_conv_with_fused_shortcut(cuda, split):
    NB, H, W, Cin, Cout, Csc = 2, 8, 16, 128, 64, 192
    g = torch.Generator(device="cpu").manual_seed(9)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    xs = torch.randn(NB, Csc, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    ws = (torch.randn(Cout, Csc, 1, 1, generator=g) / math.sqrt(Csc)).to(cuda)
    bs = torch.randn(Cout, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=split, device=cuda, sc_w=ws, sc_b=bs)
    if split:
        a, s = to_split(nhwc_rows(x)), to_split(nhwc_rows(xs))
        ref = F.conv2d(x.double(), w.double(), b.double(), padding=1) + F.conv2d(xs.double(), ws.double(), bs.double())
        ref = ref.float()
    else:
        a, s = bf(nhwc_rows(x)), bf(nhwc_rows(xs))
        ref = F.conv2d(bf(x).float(), bf(w).float(), b, padding=1) + F.conv2d(bf(xs).float(), bf(ws).float(), bs)
    of = torch.empty(NB * H * W, Cout, device=cuda)
    ops.run_conv(pc, a, NB, H, W, sc_x=s, out_f32=of)
    torch.cuda.synchronize()
    assert rel_err(of, nhwc_rows(ref)) < 3e-5


@pytest.mark.parametrize("k,dil,C,Lx", [(3, 1, 64, 1000), (7, 3, 128, 517), (11, 5, 64, 2049), (7, 1, 32, 700)])
def test_conv1d_dilated(cuda, k, dil, C, Lx):
    B = 2
    g = torch.Generator(device="cpu").manual_seed(k * 10 + dil)
    x = torch.randn(B, C, Lx, generator=g).to(cuda)
    w = (torch.randn(C, C, k, generator=g) / math.sqrt(k * C)).to(cuda)
    b = torch.randn(C, generator=g).to(cuda)
    res = torch.randn(B * Lx, C, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=False, device=cuda, dilation=dil)
    xb = bf(x.permute(0, 2, 1).reshape(B * Lx, C).contiguous())
    of = torch.empty(B * Lx, C, device=cuda)
    ob = torch.empty(B * Lx, C, device=cuda, dtype=torch.bfloat16)
    ops.run_conv(pc, xb, B, 1, Lx, res=res, out_f32=of, out_bf16=ob, act=L.ACT_LRELU, act_param=0.1)
    ref = F.conv1d(bf(x).float(), bf(w).float(), b, padding=(k * dil - dil) // 2, dilation=dil)
    ref = ref.permute(0, 2, 1).reshape(B * Lx, C) + res
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 2e-5
    assert rel_err(ob, F.leaky_relu(ref, 0.1)) < 5e-3
    # accumulate: out += x * alpha
    of2 = of.clone()
    ops.run_conv(pc, xb, B, 1, Lx, res=res, out_f32=of2, alpha=1.0 / 3, accumulate=True)
    torch.cuda.synchronize()
    assert rel_err(of2, ref + ref / 3) < 2e-5


@pytest.mark.parametrize("bn", [128, 256])
def test_geglu_epilogue(cuda, bn):
    M, Cc = 520, 128
    inner = 4 * Cc
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(M, Cc, generator=g).to(cuda)
    w = (torch.randn(2 * inner, Cc, generator=g) / math.sqrt(Cc)).to(cuda)
    b = torch.randn(2 * inner, generator=g).to(cuda)
    pc = ops.PackedConv(w, b, split=False, device=cuda, geglu_bn=bn)
    xb = bf(x)
    ob = torch.empty(M, inner, device=cuda, dtype=torch.bfloat16)
    ops.run_linear(pc, xb, out_bf16=ob)
    proj = xb.float() @ bf(w).float().t() + b
    ref = proj[:, :inner] * F.gelu(proj[:, inner:])
    torch.cuda.synchronize()
    assert rel_err(ob, ref) < 5e-3


def attn_ref(q, k, v, heads, scale, bias=None):
    B, Lq, Cc = q.shape
    Lk = k.shape[1]
    d = Cc // heads
    qh = q.view(B, Lq, heads, d).transpose(1, 2)
    kh = k.view(B, Lk, heads, d).transpose(1, 2)
    vh = v.view(B, Lk, heads, d).transpose(1, 2)
    s = qh @ kh.transpose(-1, -2) * scale
    if bias is not None:
        s = s + bias[:, None, None, :]
    p = s.softmax(-1)
    return (p @ vh).transpose(1, 2).reshape(B, Lq, Cc)


@pytest.mark.parametrize("B,heads,Lq,Lk,masked", [(2, 2, 300, 300, False), (1, 5, 4096, 4096, False),
                                                   (2, 4, 200, 64, True), (3, 1, 8, 8, False), (2, 2, 130, 77, True)])
def test_attention(cuda, B, heads, Lq, Lk, masked):
    Cc = heads * 64
    g = torch.Generator(device="cpu").manual_seed(Lq + Lk)
    q = torch.randn(B, Lq, Cc, generator=g).to(cuda)
    k = torch.randn(B, Lk, Cc, generator=g).to(cuda)
    v = torch.randn(B, Lk, Cc, generator=g).to(cuda)
    bias = None
    if masked:
        m = torch.rand(B, Lk, generator=g) > 0.3
        m[:, 0] = True
        bias = ((1 - m.float()) * -10000.0).to(cuda)
    # fused QKV-style buffers: q in its own matrix, k|v side by side
    qb = bf(q).reshape(B * Lq, Cc).contiguous()
    kvb = torch.cat([bf(k), bf(v)], dim=-1).reshape(B * Lk, 2 * Cc).contiguous()
    out = torch.zeros(B * Lq, Cc, device=cuda, dtype=torch.bfloat16)
    L.attention(qb, kvb, kvb, out, batch=B, heads=heads, Lq=Lq, Lk=Lk, scale=0.125, k_col0=0, v_col0=Cc, kbias=bias)
    ref = attn_ref(bf(q).float(), bf(k).float(), bf(v).float(), heads, 0.125, bias)
    torch.cuda.synchronize()
    assert rel_err(out.view(B, Lq, Cc), ref) < 1e-2


def test_attention_split_matches_fp32(cuda):
    B, heads, Lq, Lk = 2, 2, 260, 260
    Cc = heads * 64
    g = torch.Generator(device="cpu").manual_seed(21)
    q = torch.randn(B * Lq, Cc, generator=g).to(cuda)
    k = torch.randn(B * Lk, Cc, generator=g).to(cuda)
    v = torch.randn(B * Lk, Cc, generator=g).to(cuda)
    qs, ks, vs = to_split(q), to_split(k), to_split(v)
    out = torch.zeros(B * Lq, 2 * Cc, device=cuda, dtype=torch.bfloat16)
    L.attention(qs, ks, vs, out, batch=B, heads=heads, Lq=Lq, Lk=Lk, scale=0.125, nsplit=2, q_lo_off=Cc, k_lo_off=Cc,
                v_lo_off=Cc, split_off=Cc)
    ref = attn_ref(q.double().view(B, Lq, Cc), k.double().view(B, Lk, Cc), v.double().view(B, Lk, Cc), heads, 0.125)
    torch.cuda.synchronize()
    rec = out[:, :Cc].float() + out[:, Cc:].float()
    assert rel_err(rec.view(B, Lq, Cc), ref.float()) < 5e-5


@pytest.mark.parametrize("C0,C1,act,eps", [(320, 0, L.ACT_SILU, 1e-5), (640, 320, L.ACT_SILU, 1e-5),
                                           (64, 0, L.ACT_NONE, 1e-6), (128, 64, L.ACT_SILU, 1e-6)])
def test_groupnorm(cuda, C0, C1, act, eps):
    NB, HW = 3, 200
    g = torch.Generator(device="cpu").manual_seed(C0 + C1)
    x0 = (torch.randn(NB * HW, C0, generator=g) * 2 + 0.5).to(cuda)
    x1 = bf(torch.randn(NB * HW, C1, generator=g)).to(cuda) if C1 else None
    Cc = C0 + C1
    gamma = torch.randn(Cc, generator=g).to(cuda)
    beta = torch.randn(Cc, generator=g).to(cuda)
    st0 = torch.zeros(NB, C0, 2, device=cuda, dtype=torch.float64)
    st1 = torch.zeros(NB, C1, 2, device=cuda, dtype=torch.float64) if C1 else None
    L.groupnorm_stats(x0, NB, HW, st0)                     # the stand-alone per-channel statistics pass
    if C1:
        L.groupnorm_stats(x1, NB, HW, st1)
    assert rel_err(st0[..., 0].float(), x0.view(NB, HW, C0).sum(1)) < 1e-5
    y = torch.empty(NB * HW, 2 * Cc, device=cuda, dtype=torch.bfloat16)
    raw = torch.empty(NB * HW, 2 * Cc, device=cuda, dtype=torch.bfloat16)
    L.groupnorm(x0, st0, x1, st1, NB, HW, 32, gamma, beta, eps, act, y, split_off=Cc, raw=raw, raw_split_off=Cc)
    xc = x0 if x1 is None else torch.cat([x0, x1.float()], dim=1)
    ref = F.group_norm(xc.view(NB, HW, Cc).permute(0, 2, 1).double(), 32, gamma.double(), beta.double(), eps)
    if act == L.ACT_SILU:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1).reshape(NB * HW, Cc).float()
    torch.cuda.synchronize()
    assert rel_err(y[:, :Cc].float() + y[:, Cc:].float(), ref) < 2e-5
    assert rel_err(y[:, :Cc], ref) < 5e-3
    assert rel_err(raw[:, :Cc].float() + raw[:, Cc:].float(), xc) < 1e-5


# NB, H, W, Cin, Cout, taps, (plan, launches) with an fp32 output and with a bf16-only output; plan = (block_n, mode,
# ksplit), launches 1 = statistics from the epilogue, 2 = pass after the GEMM
@pytest.mark.parametrize("shape", [(16, 8, 4, 128, 320, 1, ((160, 1, 1), 1), ((160, 1, 1), 1)),     # full tiles
                                   (4, 16, 16, 64, 640, 9, ((128, 1, 1), 1), ((128, 1, 1), 1)),     # 3x3, full tiles
                                   (3, 4, 8, 64, 64, 9, ((64, 1, 1), 2), ((64, 1, 1), 2)),          # partial tiles
                                   # under-filled: split-K with the fp32 output, full N tiles of 128 with bf16 only
                                   (2, 2, 32, 1280, 1280, 9, ((160, 1, 2), 2), ((128, 1, 1), 1))])
def test_conv_gemm_emits_groupnorm_statistics(cuda, monkeypatch, shape):
    """tng_conv_gemm(gn_stats=...): per-(image, channel) sum / sum of squares of the fp32 output, accumulated from the
    epilogue (or by the follow-up pass when tiles are partial / split-K), must equal the column sums of what was stored."""
    NB, H, W, Cin, Cout, taps, plan_f32, plan_bf16 = shape
    g = torch.Generator(device="cpu").manual_seed(Cout + taps)
    k = 3 if taps == 9 else 1
    w = torch.randn(Cout, Cin, k, k, generator=g) * (Cin * taps) ** -0.5
    b = torch.randn(Cout, generator=g)
    x = torch.randn(NB * H * W, Cin, generator=g)
    res = torch.randn(NB * H * W, Cout, generator=g).to(cuda)
    pc = PackedConv(w if k == 3 else w[:, :, 0, 0], b, split=False, device=cuda)
    out = torch.zeros(NB * H * W, Cout, device=cuda)
    st = torch.zeros(NB, Cout, 2, device=cuda, dtype=torch.float64)
    got = run_conv_planned(monkeypatch, pc, bf(x).to(cuda), NB, H, W, res=res if taps == 1 else None, out_f32=out,
                           gn_stats=st, stats_hw=H * W)
    assert got == plan_f32
    torch.cuda.synchronize()
    o = out.double().view(NB, H * W, Cout)
    assert rel_err(st[..., 0], o.sum(1)) < 1e-6 and rel_err(st[..., 1], (o * o).sum(1)) < 1e-6
    # accumulators ADD: a second launch doubles them
    run_conv(pc, bf(x).to(cuda), NB, H, W, res=res if taps == 1 else None, out_f32=out, gn_stats=st, stats_hw=H * W)
    torch.cuda.synchronize()
    assert rel_err(st[..., 0], 2 * o.sum(1)) < 1e-6
    # bf16-only output (conv1 of a resnet in perf mode): the statistics are those of the fp32 epilogue values when they
    # ride in the epilogue, of the stored bf16 values when the follow-up pass computes them — either way within bf16
    # rounding of the fp32 sums
    ob = torch.zeros(NB * H * W, Cout, device=cuda, dtype=torch.bfloat16)
    st2 = torch.zeros(NB, Cout, 2, device=cuda, dtype=torch.float64)
    got = run_conv_planned(monkeypatch, pc, bf(x).to(cuda), NB, H, W, res=res if taps == 1 else None, out_bf16=ob,
                           gn_stats=st2, stats_hw=H * W)
    assert got == plan_bf16
    torch.cuda.synchronize()
    assert rel_err(ob, out) < 5e-3
    assert rel_err(st2[..., 1], (o * o).sum(1)) < 5e-3 and rel_err(st2[..., 0], o.sum(1)) < 2e-2


@pytest.mark.parametrize("B,Lq,spread", [(2, 256, 1.0), (1, 1024, 1.0), (2, 384, 6.0)])
def test_attention_wide_d512(cuda, B, Lq, spread):
    """tng_attention_wide (the VAE AttnBlock: one head of width 512, flash-style) against torch; `spread` > 1 makes the
    key magnitudes grow along the sequence so that rows outgrow the lazy-rescale threshold (O rescale in TMEM)."""
    Cc = 512
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + Lq)
    q = torch.randn(B, Lq, Cc, generator=g)
    k = torch.randn(B, Lq, Cc, generator=g) * torch.linspace(1.0, spread, Lq)[None, :, None]
    v = torch.randn(B, Lq, Cc, generator=g)
    qkv = torch.cat([bf(q), bf(k), bf(v)], dim=-1).reshape(B * Lq, 3 * Cc).contiguous().to(cuda)
    out = torch.zeros(B * Lq, Cc, device=cuda, dtype=torch.bfloat16)
    L.attention_wide(qkv, qkv, qkv, out, batch=B, L=Lq, dim=Cc, scale=Cc ** -0.5, q_col0=0, k_col0=Cc, v_col0=2 * Cc)
    s = (bf(q).double() @ bf(k).double().transpose(1, 2)) * Cc ** -0.5
    ref = (s.softmax(-1) @ bf(v).double()).float()
    torch.cuda.synchronize()
    assert rel_err(out.view(B, Lq, Cc).cpu(), ref) < 1e-2      # P and the output are rounded to bf16
    with pytest.raises(L.TangoB200Error):
        L.attention_wide(qkv, qkv, qkv, out, batch=B, L=Lq - 64, dim=Cc, scale=1.0)


@pytest.mark.parametrize("Cc", [64, 320, 1280])
def test_layernorm(cuda, Cc):
    rows = 777
    g = torch.Generator(device="cpu").manual_seed(Cc)
    x = (torch.randn(rows, Cc, generator=g) * 3 + 1).to(cuda)
    gamma = torch.randn(Cc, generator=g).to(cuda)
    beta = torch.randn(Cc, generator=g).to(cuda)
    y = torch.empty(rows, 2 * Cc, device=cuda, dtype=torch.bfloat16)
    L.layernorm(x, gamma, beta, 1e-5, y, split_off=Cc)
    ref = F.layer_norm(x, (Cc,), gamma, beta, 1e-5)
    torch.cuda.synchronize()
    assert rel_err(y[:, :Cc].float() + y[:, Cc:].float(), ref) < 1e-5


def test_cast_upsample_softmax_transpose(cuda):
    g = torch.Generator(device="cpu").manual_seed(1)
    NB, H, W, Cc = 2, 6, 4, 64
    x = torch.randn(NB * H * W, Cc, generator=g).to(cuda)
    y = torch.empty(NB * 4 * H * W, Cc, device=cuda, dtype=torch.bfloat16)
    L.cast_act(x, NB, H, W, y, upsample2x=True, act=L.ACT_LRELU, act_param=0.1)
    ref = F.interpolate(F.leaky_relu(x, 0.1).view(NB, H, W, Cc).permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    torch.cuda.synchronize()
    assert torch.equal(y, bf(ref.permute(0, 2, 3, 1).reshape(-1, Cc)))
    s = torch.randn(50, 1000, generator=g).to(cuda) * 5
    p = torch.empty(50, 1024, device=cuda, dtype=torch.bfloat16)
    L.softmax_rows(s, 0.3, p, L=1000)
    torch.cuda.synchronize()
    assert rel_err(p[:, :1000], (s * 0.3).softmax(-1)) < 5e-3
    t = bf(torch.randn(3, 70, 96, generator=g)).to(cuda)
    tt = torch.empty(3 * 96, 70, device=cuda, dtype=torch.bfloat16)
    L.transpose_bf16(t.view(3 * 70, 96), 3, 70, 96, tt)
    torch.cuda.synchronize()
    assert torch.equal(tt.view(3, 96, 70), t.transpose(1, 2))


def test_small_fp32_ops(cuda):
    g = torch.Generator(device="cpu").manual_seed(2)
    t = torch.tensor([0.0, 1.0, 995.0, 500.0], device=cuda)
    out = torch.empty(4, 320, device=cuda)
    L.timestep_embedding(t, 320, True, 0.0, out)
    half = 160
    ex = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device=cuda) / half)
    e = t[:, None] * ex[None]
    ref = torch.cat([torch.cos(e), torch.sin(e)], -1)
    torch.cuda.synchronize()
    assert (out - ref).abs().max().item() < 2e-4
    x = torch.randn(5, 320, generator=g).to(cuda)
    w = torch.randn(1280, 320, generator=g).to(cuda) / 18
    b = torch.randn(1280, generator=g).to(cuda)
    y = torch.empty(5, 1280, device=cuda)
    L.linear_f32(x, w, b, y, pre_act=L.ACT_SILU, post_act=L.ACT_NONE)
    torch.cuda.synchronize()
    assert rel_err(y, F.linear(F.silu(x), w, b)) < 1e-5
    # ConvTranspose1d via GEMM + gather
    B, Cin, Cout, Lin, k, u = 2, 64, 32, 37, 16, 5
    xin = torch.randn(B, Cin, Lin, generator=g).to(cuda)
    wt = (torch.randn(Cin, Cout, k, generator=g) / 10).to(cuda)
    bt = torch.randn(Cout, generator=g).to(cuda)
    pad = (k - u) // 2
    ref = F.conv_transpose1d(bf(xin).float(), bf(wt).float(), bt, stride=u, padding=pad)
    Lout = ref.shape[-1]
    wg = wt.permute(2, 1, 0).reshape(k * Cout, Cin)  # row (t, co)
    pc = ops.PackedConv(wg, None, split=False, device=cuda)
    Y = torch.empty(B * Lin, k * Cout, device=cuda)
    ops.run_conv(pc, bf(xin.permute(0, 2, 1).reshape(B * Lin, Cin).contiguous()), B, 1, Lin, out_f32=Y)
    yo = torch.empty(B * Lout, Cout, device=cuda)
    L.convt_gather(Y, B, Lin, k, Cout, u, pad, Lout, bt, yo)
    torch.cuda.synchronize()
    assert rel_err(yo.view(B, Lout, Cout), ref.permute(0, 2, 1)) < 2e-5
    xw = torch.tensor([0.0, 0.5, -0.5, 20.0, -20.0, 1e-3], device=cuda)
    wf = torch.empty(6, device=cuda)
    wi = torch.empty(6, device=cuda, dtype=torch.int16)
    L.tanh_to_i16(xw, 6, 1, wf, wi)
    torch.cuda.synchronize()
    import numpy as np
    expect = (torch.tanh(xw).cpu().numpy() * 32768).astype("int16")
    assert np.array_equal(wi.cpu().numpy(), expect)


# ------------------------------------------------------------------------------------------------ T5 front-end kernels
@pytest.mark.parametrize("Cc", [128, 1024, 2048])
def test_rmsnorm(cuda, Cc):
    rows = 333
    g = torch.Generator(device="cpu").manual_seed(Cc)
    x = (torch.randn(rows, Cc, generator=g) * 3 + 0.5).to(cuda)
    gamma = torch.randn(Cc, generator=g).to(cuda)
    y = torch.empty(rows, 2 * Cc, device=cuda, dtype=torch.bfloat16)
    yf = torch.empty(rows, Cc, device=cuda)
    L.rmsnorm(x, gamma, 1e-6, y, split_off=Cc, y_f32=yf)
    ref = gamma * (x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-6))
    torch.cuda.synchronize()
    assert rel_err(yf, ref) < 1e-6
    assert rel_err(y[:, :Cc].float() + y[:, Cc:].float(), ref) < 1e-5


def test_gather_rows(cuda):
    g = torch.Generator(device="cpu").manual_seed(5)
    table = torch.randn(97, 128, generator=g).to(cuda)
    ids = torch.randint(0, 97, (41,), generator=g).to(cuda)
    out = torch.empty(41, 128, device=cuda)
    L.gather_rows(table, ids, out)
    torch.cuda.synchronize()
    assert torch.equal(out, table[ids])


@pytest.mark.parametrize("B,heads,Lt", [(2, 2, 10), (3, 16, 64), (1, 4, 150), (1, 2, 513)])
def test_rel_attention(cuda, B, heads, Lt):
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + Lt)
    inner = heads * 64
    qkv = torch.randn(B * Lt, 3 * inner, generator=g)
    qkv[:, :inner] *= 0.3
    relbias = torch.randn(heads, 2 * Lt - 1, generator=g)
    mask = torch.ones(B, Lt)
    mask[0, max(1, Lt - 3):] = 0
    kbias = (1.0 - mask) * torch.finfo(torch.float32).min
    out = torch.empty(B * Lt, 2 * inner, device=cuda, dtype=torch.bfloat16)
    L.rel_attention(qkv.to(cuda), relbias.to(cuda), kbias.to(cuda), out, batch=B, heads=heads, L=Lt, q_col0=0,
                    k_col0=inner, v_col0=2 * inner, split_off=inner)
    q, k, v = (qkv[:, i * inner:(i + 1) * inner].view(B, Lt, heads, 64).transpose(1, 2) for i in range(3))
    pos = torch.arange(Lt)
    bias = relbias[:, (pos[None, :] - pos[:, None]) + Lt - 1][None] + kbias[:, None, None, :]
    ref = ((q @ k.transpose(-1, -2) + bias).softmax(-1) @ v).transpose(1, 2).reshape(B * Lt, inner)
    torch.cuda.synchronize()
    got = out[:, :inner].float() + out[:, inner:].float()
    assert rel_err(got.cpu(), ref) < 2e-5


def test_gated_tanh_gelu_epilogue(cuda):
    M, Cc, inner = 70, 128, 256
    g = torch.Generator(device="cpu").manual_seed(9)
    x = torch.randn(M, Cc, generator=g).to(cuda)
    w = (torch.randn(2 * inner, Cc, generator=g) * 2 / math.sqrt(Cc)).to(cuda)     # rows: [hidden | gate]
    pc = ops.PackedConv(w, None, split=False, device=cuda, geglu_bn=256, geglu_tanh=True)
    xb = bf(x)
    ob = torch.empty(M, inner, device=cuda, dtype=torch.bfloat16)
    ops.run_linear(pc, xb, out_bf16=ob)
    proj = xb.float() @ bf(w).float().t()
    ref = proj[:, :inner] * F.gelu(proj[:, inner:], approximate="tanh")
    torch.cuda.synchronize()
    assert rel_err(ob, ref) < 5e-3
    # split (parity) mode: ~fp32 accuracy
    pcs = ops.PackedConv(w, None, split=True, device=cuda, geglu_bn=256, geglu_tanh=True)
    obs = torch.empty(M, 2 * inner, device=cuda, dtype=torch.bfloat16)
    ops.run_linear(pcs, to_split(x), out_bf16=obs)
    proj = x @ w.t()
    ref = proj[:, :inner] * F.gelu(proj[:, inner:], approximate="tanh")
    torch.cuda.synchronize()
    assert rel_err(obs[:, :inner].float() + obs[:, inner:].float(), ref) < 5e-5


@pytest.mark.parametrize("NB,H,W,Cin,Cout,sc", [(16, 32, 2, 1280, 1280, 0), (5, 32, 2, 640, 320, 0), (16, 32, 2, 1280, 1280, 640)])
def test_conv3x3_underfilled_split_k(cuda, monkeypatch, NB, H, W, Cin, Cout, sc):
    """Under-filled launches with a long reduction (the 32x2 level of the UNet) take the split-K path: two CTAs per
    output tile red.add their fp32 partials into a zeroed output; bias / time vector / residual enter once; a fused
    1x1 shortcut rides along as an extra k-group. The 5-image case has a ragged last M tile."""
    g = torch.Generator(device="cpu").manual_seed(NB + Cin + sc)
    x = torch.randn(NB, Cin, H, W, generator=g).to(cuda)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    b = torch.randn(Cout, generator=g).to(cuda)
    temb = torch.randn(NB, Cout, generator=g).to(cuda)
    xb = bf(nhwc_rows(x))
    of = torch.full((NB * H * W, Cout), float("nan"), device=cuda)
    if sc:
        xs = torch.randn(NB, sc, H, W, generator=g).to(cuda)
        ws = (torch.randn(Cout, sc, 1, 1, generator=g) / math.sqrt(sc)).to(cuda)
        bs = torch.randn(Cout, generator=g).to(cuda)
        pc = ops.PackedConv(w, b, split=False, device=cuda, sc_w=ws, sc_b=bs)
        plan, _ = run_conv_planned(monkeypatch, pc, xb, NB, H, W, sc_x=bf(nhwc_rows(xs)), rowvec=temb, out_f32=of)
        ref = F.conv2d(bf(x).float(), bf(w).float(), b, padding=1) + temb[:, :, None, None]
        ref = nhwc_rows(ref + F.conv2d(bf(xs).float(), bf(ws).float(), bs))
    else:
        res = torch.randn(NB * H * W, Cout, generator=g).to(cuda)
        pc = ops.PackedConv(w, b, split=False, device=cuda)
        plan, _ = run_conv_planned(monkeypatch, pc, xb, NB, H, W, rowvec=temb, res=res, alpha=0.5, out_f32=of)
        ref = F.conv2d(bf(x).float(), bf(w).float(), b, padding=1) + temb[:, :, None, None]
        ref = (nhwc_rows(ref) + res) * 0.5
    assert plan == (160, 1, 2)
    torch.cuda.synchronize()
    assert rel_err(of, ref) < 2e-5
    of2 = torch.full_like(of, float("nan"))
    if sc:
        ops.run_conv(pc, xb, NB, H, W, sc_x=bf(nhwc_rows(xs)), rowvec=temb, out_f32=of2)
    else:
        ops.run_conv(pc, xb, NB, H, W, rowvec=temb, res=res, alpha=0.5, out_f32=of2)
    torch.cuda.synchronize()
    assert torch.equal(of, of2)     # two partials per element: order-independent, run-to-run identical

