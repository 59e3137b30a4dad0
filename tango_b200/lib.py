"""ctypes binding of libtango_b200.so (include/tango_b200.h) + thin torch-tensor helpers.

PyTorch is plumbing only here: it owns device memory and the current CUDA stream; every compute call goes
through the C ABI into the hand-written sm_100a kernels. There is no CPU / eager fallback: if the library is
missing or a call fails, a TangoB200Error is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

from . import build as _build

ACT_NONE, ACT_SILU, ACT_LRELU, ACT_GEGLU, ACT_GEGLU_TANH = 0, 1, 2, 3, 4
DT_F32, DT_BF16 = 0, 1
MAX_AVIEWS, MAX_KGROUPS = 4, 40

# every symbol include/tango_b200.h declares (tests/test_cabi.py checks the exports against the header)
SYMBOLS = [
    "tng_version", "tng_last_error", "tng_launch_count", "tng_conv_gemm", "tng_attention",
    "tng_groupnorm_stats", "tng_groupnorm_apply", "tng_layernorm", "tng_cast_act", "tng_softmax_rows",
    "tng_transpose_bf16", "tng_sched_step", "tng_timestep_embedding", "tng_linear_f32", "tng_convt_gather",
    "tng_tanh_to_i16", "tng_rmsnorm", "tng_gather_rows", "tng_rel_attention", "tng_stft_frames", "tng_stft_magnitude",
    "tng_log_clamp", "tng_attention_wide", "tng_gemm_plan", "tng_sched_multistep",
]


class TangoB200Error(RuntimeError):
    pass


class AView(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("C", C.c_int64), ("W", C.c_int64), ("H", C.c_int64), ("NB", C.c_int64),
                ("s_w", C.c_int64), ("s_h", C.c_int64), ("s_n", C.c_int64)]


class KGroup(C.Structure):
    _fields_ = [("view", C.c_int32), ("a_c0", C.c_int32), ("dw", C.c_int32), ("dh", C.c_int32),
                ("b_k0", C.c_int32), ("nkb", C.c_int32)]


class GemmDesc(C.Structure):
    _fields_ = [
        ("a", AView * MAX_AVIEWS), ("n_aviews", C.c_int32),
        ("b", C.c_void_p), ("Ncols", C.c_int64), ("Ktot", C.c_int64), ("ldb", C.c_int64),
        ("W", C.c_int32), ("H", C.c_int32), ("NB", C.c_int32),
        ("g", KGroup * MAX_KGROUPS), ("n_groups", C.c_int32),
        ("bias", C.c_void_p), ("rowvec", C.c_void_p), ("rowvec_ld", C.c_int64), ("res", C.c_void_p), ("res_dtype", C.c_int32),
        ("ldr", C.c_int64), ("alpha", C.c_float), ("accumulate", C.c_int32),
        ("out_f32", C.c_void_p), ("ld_f32", C.c_int64), ("out_bf16", C.c_void_p), ("ld_bf16", C.c_int64),
        ("act", C.c_int32), ("act_param", C.c_float), ("split_off", C.c_int32), ("block_n", C.c_int32),
        ("gn_stats", C.c_void_p), ("stats_hw", C.c_int64),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ld_q", C.c_int64), ("q_col0", C.c_int32), ("q_lo_off", C.c_int32),
        ("k", C.c_void_p), ("ld_k", C.c_int64), ("k_col0", C.c_int32), ("k_lo_off", C.c_int32),
        ("v", C.c_void_p), ("ld_v", C.c_int64), ("v_col0", C.c_int32), ("v_lo_off", C.c_int32),
        ("kbias", C.c_void_p), ("out", C.c_void_p), ("ld_o", C.c_int64), ("split_off", C.c_int32),
        ("batch", C.c_int32), ("heads", C.c_int32), ("Lq", C.c_int32), ("Lk", C.c_int32),
        ("scale", C.c_float), ("nsplit", C.c_int32),
    ]


_lib: Optional[C.CDLL] = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen libtango_b200.so (building it in-tree first if it is absent and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise TangoB200Error(f"{path} is missing: run `python -m tango_b200.build`")
        _build.build()
    lib = C.CDLL(path)
    lib.tng_version.restype = C.c_int
    lib.tng_last_error.restype = C.c_char_p
    lib.tng_launch_count.restype = C.c_uint64
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    sigs = {
        "tng_conv_gemm": [C.POINTER(GemmDesc), vp],
        "tng_gemm_plan": [C.POINTER(GemmDesc), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)],
        "tng_attention": [C.POINTER(AttnDesc), vp],
        "tng_groupnorm_stats": [vp, i32, i64, i64, i64, i64, vp, vp],
        "tng_groupnorm_apply": [vp, i32, i64, vp, vp, i32, i64, vp, i64, i64, i32, vp, vp, f32, i32, vp, i64, i32, vp,
                                i64, i32, vp],
        "tng_layernorm": [vp, i64, i64, vp, vp, f32, vp, i64, i32, vp],
        "tng_rmsnorm": [vp, i64, i64, vp, f32, vp, i64, i32, vp, vp],
        "tng_gather_rows": [vp, i64, vp, i64, i64, vp, vp],
        "tng_rel_attention": [vp, i64, i32, i32, i32, i32, i32, i32, vp, vp, vp, i64, i32, vp],
        "tng_cast_act": [vp, i64, i64, i64, i64, i64, i32, i32, f32, vp, i64, i32, vp],
        "tng_softmax_rows": [vp, i64, i64, i64, f32, vp, i64, i32, vp],
        "tng_transpose_bf16": [vp, i64, i64, i64, i64, vp, i64, vp],
        "tng_sched_step": [vp, i64, i32, f32, vp, vp, vp, vp, vp, i64, i32, i64, i64, i64, vp],
        "tng_sched_multistep": [vp, i64, i32, f32, vp, vp, vp, vp, i32, vp, vp, vp, i64, i32, i64, i64, i64, vp],
        "tng_timestep_embedding": [vp, i64, i32, i32, f32, vp, vp],
        "tng_linear_f32": [vp, i64, i64, vp, vp, i64, i32, i32, vp, vp],
        "tng_convt_gather": [vp, i64, i64, i32, i64, i32, i32, i64, vp, vp, vp],
        "tng_tanh_to_i16": [vp, i64, i64, vp, vp, vp],
        "tng_stft_frames": [vp, i64, i64, i32, vp, vp, i64, vp],
        "tng_stft_magnitude": [vp, i64, i32, i64, vp, i64, i32, vp, vp, f32, vp],
        "tng_log_clamp": [vp, i64, f32, vp, vp],
        "tng_attention_wide": [vp, i64, i32, vp, i64, i32, vp, i64, i32, vp, i64, i32, i32, i32, f32, vp],
    }
    for name, argt in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argt
        fn.restype = C.c_int
    _lib = lib
    return lib


class _Profiler:
    """Optional per-launch CUDA-event timing (bench.py's roofline leg). Off by default: zero overhead."""

    def __init__(self):
        self.enabled = False
        self.records = []  # (family, algorithmic flops, algorithmic bytes, start event, end event)

    def start(self):
        self.records = []
        self.enabled = True

    def stop(self):
        self.enabled = False
        torch.cuda.synchronize()
        out = {}
        for fam, fl, by, e0, e1 in self.records:
            d = out.setdefault(fam, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["launches"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += fl
            d["bytes"] += by
        self.records = []
        return out

    def timed(self, family, flops, nbytes, fn):
        """Run fn() (one kernel launch); when profiling, bracket it with CUDA events on the current stream."""
        if not self.enabled:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        self.records.append((family, float(flops), float(nbytes), e0, e1))
        return r


PROF = _Profiler()

def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().tng_last_error().decode("utf-8", "replace")
        raise TangoB200Error(f"{what or 'tng call'} failed ({rc}): {msg}")


def _call(family: str, nbytes: float, fn, *args) -> None:
    """One C-ABI launch; `nbytes` = its algorithmic HBM bytes (bench.py's per-family HBM roofline)."""
    PROF.timed(family, 0.0, nbytes, lambda: check(fn(*args), family))


def _esz(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.element_size()


def launch_count() -> int:
    return int(load().tng_launch_count())


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return DT_F32
    if t.dtype == torch.bfloat16:
        return DT_BF16
    raise TangoB200Error(f"unsupported dtype {t.dtype}")


def require_cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise TangoB200Error("tango_b200 kernels need CUDA tensors (there is no CPU fallback)")


def require_cuda_device(device) -> None:
    """Models refuse to pack / run anywhere but on a CUDA device (there is no CPU fallback)."""
    if torch.device(device).type != "cuda":
        raise TangoB200Error("tango_b200 runs on CUDA only: call .to('cuda') (there is no CPU fallback)")


# --------------------------------------------------------------------------------------------------- conv / gemm
class View:
    """A bf16 channels-last activation view (img, h, w, c) with element strides."""

    __slots__ = ("t", "C", "W", "H", "NB", "s_w", "s_h", "s_n", "off")

    def __init__(self, t: torch.Tensor, C_: int, W: int, H: int, NB: int, s_w: int, s_h: int, s_n: int, off: int = 0):
        self.t, self.C, self.W, self.H, self.NB = t, C_, W, H, NB
        self.s_w, self.s_h, self.s_n, self.off = s_w, s_h, s_n, off

    @staticmethod
    def rows(t: torch.Tensor, NB: int, H: int, W: int, C_: Optional[int] = None) -> "View":
        """t: contiguous bf16 [NB*H*W, ld]; the view exposes its first C_ (default ld) channels."""
        ld = t.shape[-1]
        return View(t, ld if C_ is None else C_, W, H, NB, ld, W * ld, H * W * ld)


def _gemm_desc(views: Sequence[View], groups: Sequence[tuple], weight: torch.Tensor, W: int, H: int, NB: int, *,
               bias=None, rowvec=None, res=None, alpha: float = 1.0, accumulate: bool = False, out_f32=None,
               out_bf16=None, act: int = ACT_NONE, act_param: float = 0.0, split_off: int = 0, block_n: int = 0,
               ld_f32: Optional[int] = None, ld_bf16: Optional[int] = None, ldr: Optional[int] = None,
               rowvec_ld: int = 0, gn_stats: Optional[torch.Tensor] = None, stats_hw: int = 0) -> GemmDesc:
    d = GemmDesc()
    require_cuda(weight, bias, rowvec, res, out_f32, out_bf16)
    assert weight.dtype == torch.bfloat16 and weight.stride(1) == 1
    d.n_aviews = len(views)
    for i, v in enumerate(views):
        require_cuda(v.t)
        assert v.t.dtype == torch.bfloat16
        d.a[i] = AView(v.t.data_ptr() + 2 * v.off, v.C, v.W, v.H, v.NB, v.s_w, v.s_h, v.s_n)
    d.b = weight.data_ptr()
    d.Ncols, d.Ktot = weight.shape
    d.ldb = weight.stride(0)
    d.W, d.H, d.NB = W, H, NB
    d.n_groups = len(groups)
    if len(groups) > MAX_KGROUPS:
        raise TangoB200Error(f"{len(groups)} k-groups > {MAX_KGROUPS}")
    for i, g in enumerate(groups):
        d.g[i] = KGroup(*g)
    d.bias = ptr(bias)
    d.rowvec = ptr(rowvec)
    d.rowvec_ld = rowvec_ld
    d.res = ptr(res)
    if res is not None:
        d.res_dtype = _dt(res)
        d.ldr = res.stride(0) if ldr is None else ldr
    d.alpha = alpha
    d.accumulate = int(accumulate)
    d.out_f32 = ptr(out_f32)
    if out_f32 is not None:
        d.ld_f32 = out_f32.stride(0) if ld_f32 is None else ld_f32
    d.out_bf16 = ptr(out_bf16)
    if out_bf16 is not None:
        d.ld_bf16 = out_bf16.stride(0) if ld_bf16 is None else ld_bf16
    d.act, d.act_param, d.split_off, d.block_n = act, act_param, split_off, block_n
    if gn_stats is not None:
        require_cuda(gn_stats)
        assert gn_stats.dtype == torch.float64 and gn_stats.is_contiguous() and stats_hw > 0
        d.gn_stats, d.stats_hw = gn_stats.data_ptr(), stats_hw
    return d


def _plan(d: GemmDesc) -> tuple:
    bn, mode, ks = C.c_int32(0), C.c_int32(0), C.c_int32(0)
    check(load().tng_gemm_plan(C.byref(d), C.byref(bn), C.byref(mode), C.byref(ks)), "tng_gemm_plan")
    return bn.value, mode.value, ks.value


def gemm_plan(views: Sequence[View], groups: Sequence[tuple], weight: torch.Tensor, W: int, H: int, NB: int,
              **kw) -> tuple:
    """(block_n, mode, ksplit) that tng_conv_gemm would launch for these arguments (same signature as conv_gemm):
    the N tile, 1 = one CTA per SM / 4 = CTA pair on a 256 x 2*block_n tile, and the split-K factor."""
    kw.pop("algo_k", None)
    return _plan(_gemm_desc(views, groups, weight, W, H, NB, **kw))


def conv_gemm(views: Sequence[View], groups: Sequence[tuple], weight: torch.Tensor, W: int, H: int, NB: int, *,
              algo_k: Optional[int] = None, **kw) -> None:
    """Launch tng_conv_gemm. groups: (view, a_c0, dw, dh, b_k0, nkb). weight: bf16 [Ncols, Ktot].
    Epilogue keywords: bias, rowvec (+ rowvec_ld), res (+ ldr), alpha, accumulate, out_f32 (+ ld_f32), out_bf16
    (+ ld_bf16), act, act_param, split_off, block_n, gn_stats, stats_hw.
    algo_k: algorithmic reduction length (taps * Cin of the reference op) for the profiler's FLOP count.
    gn_stats: fp64 [images, Ncols, 2] per-channel GroupNorm accumulators of the fp32 output (zeroed by the caller),
    images of stats_hw rows each."""
    lib = load()
    d = _gemm_desc(views, groups, weight, W, H, NB, **kw)
    if PROF.enabled:
        k_alg = algo_k if algo_k is not None else sum(g[5] for g in groups) * 64
        flops = 2.0 * W * H * NB * weight.shape[0] * k_alg
        bn, mode, ks = _plan(d)
        tag = {1: "1cta", 2: "mcast", 3: "pair", 4: "pair2"}.get(mode, str(mode))
        fam = f"gemm_tc<{bn},{tag}" + (",splitk>" if ks > 1 else ">")
        PROF.timed(fam, flops, 0, lambda: check(lib.tng_conv_gemm(C.byref(d), stream_ptr()), "tng_conv_gemm"))
        return
    check(lib.tng_conv_gemm(C.byref(d), stream_ptr()), "tng_conv_gemm")


def attention(q, k, v, out, *, batch, heads, Lq, Lk, scale, q_col0=0, k_col0=0, v_col0=0, kbias=None, nsplit=1,
              q_lo_off=0, k_lo_off=0, v_lo_off=0, split_off=0) -> None:
    lib = load()
    require_cuda(q, k, v, out, kbias)
    d = AttnDesc()
    d.q, d.ld_q, d.q_col0, d.q_lo_off = q.data_ptr(), q.stride(0), q_col0, q_lo_off
    d.k, d.ld_k, d.k_col0, d.k_lo_off = k.data_ptr(), k.stride(0), k_col0, k_lo_off
    d.v, d.ld_v, d.v_col0, d.v_lo_off = v.data_ptr(), v.stride(0), v_col0, v_lo_off
    d.kbias = ptr(kbias)
    d.out, d.ld_o, d.split_off = out.data_ptr(), out.stride(0), split_off
    d.batch, d.heads, d.Lq, d.Lk, d.scale, d.nsplit = batch, heads, Lq, Lk, scale, nsplit
    PROF.timed("attention_tc", 4.0 * batch * heads * Lq * Lk * 64, 0,
               lambda: check(lib.tng_attention(C.byref(d), stream_ptr()), "tng_attention"))


def attention_wide(q, k, v, out, *, batch, L, dim, scale, q_col0=0, k_col0=0, v_col0=0) -> None:
    """One-head flash attention of width `dim` (= 512: the VAE AttnBlock); see tng_attention_wide."""
    require_cuda(q, k, v, out)
    PROF.timed("attention_wide", 4.0 * batch * L * L * dim, 0,
               lambda: check(load().tng_attention_wide(q.data_ptr(), q.stride(0), q_col0, k.data_ptr(), k.stride(0), k_col0,
                                                       v.data_ptr(), v.stride(0), v_col0, out.data_ptr(), out.stride(0),
                                                       batch, L, dim, scale, stream_ptr()), "tng_attention_wide"))


# --------------------------------------------------------------------------------------------------- norms etc.
def groupnorm_stats(x, NB, HW, stats):
    """stats fp64 [NB, C, 2] += per-channel (sum, sum of squares) of x [NB*HW, C] — the stand-alone pass for tensors whose
    statistics did not come out of the producing GEMM (conv_gemm(gn_stats=...))."""
    require_cuda(x, stats)
    Cc = x.shape[-1]
    _call("gn_stats", NB * HW * Cc * _esz(x), load().tng_groupnorm_stats, x.data_ptr(), _dt(x), Cc, x.stride(0), NB, HW,
          stats.data_ptr(), stream_ptr())


def groupnorm(x0, st0, x1, st1, NB, HW, groups, gamma, beta, eps, act, y, *, split_off=0, raw=None, raw_split_off=0):
    """GroupNorm(+act) of the channel concat [x0 | x1] (x1 may be None) -> bf16 y; optional raw bf16 copy. st0 / st1:
    the per-channel fp64 statistics [NB, C, 2] of x0 / x1."""
    lib = load()
    require_cuda(x0, x1, st0, st1, gamma, beta, y, raw)
    C0 = x0.shape[-1]
    C1 = 0 if x1 is None else x1.shape[-1]
    rows = NB * HW
    in_bytes = rows * (C0 * _esz(x0) + C1 * _esz(x1))
    out_bytes = rows * (C0 + C1) * 2 * (2 if split_off else 1) * (2 if raw is not None else 1)
    _call("gn_apply", in_bytes + out_bytes, lib.tng_groupnorm_apply, x0.data_ptr(), _dt(x0), C0, st0.data_ptr(), ptr(x1),
          0 if x1 is None else _dt(x1), C1, ptr(st1), NB, HW, groups, gamma.data_ptr(), beta.data_ptr(), eps, act,
          y.data_ptr(), y.stride(0), split_off, ptr(raw), 0 if raw is None else raw.stride(0), raw_split_off, stream_ptr())


def layernorm(x, gamma, beta, eps, y, *, split_off=0):
    require_cuda(x, gamma, beta, y)
    rows, Cc = x.shape
    _call("layernorm", rows * Cc * (4 + (4 if split_off else 2)), load().tng_layernorm, x.data_ptr(), rows, Cc,
          gamma.data_ptr(), beta.data_ptr(), eps, y.data_ptr(), y.stride(0), split_off, stream_ptr())


def rmsnorm(x, gamma, eps, y=None, *, split_off=0, y_f32=None):
    require_cuda(x, gamma)
    rows, Cc = x.shape
    check(load().tng_rmsnorm(x.data_ptr(), rows, Cc, gamma.data_ptr(), eps, y.data_ptr() if y is not None else None,
                             y.stride(0) if y is not None else 0, split_off,
                             y_f32.data_ptr() if y_f32 is not None else None, stream_ptr()), "tng_rmsnorm")


def gather_rows(table, ids, out):
    require_cuda(table, ids, out)
    if ids.dtype != torch.int64 or not ids.is_contiguous():
        raise TangoB200Error("gather_rows: ids must be a contiguous int64 tensor")
    check(load().tng_gather_rows(table.data_ptr(), table.shape[0], ids.data_ptr(), ids.numel(), table.shape[1],
                                 out.data_ptr(), stream_ptr()), "tng_gather_rows")


def rel_attention(qkv, relbias, kbias, out, *, batch, heads, L, q_col0, k_col0, v_col0, split_off=0):
    require_cuda(qkv, relbias, out)
    check(load().tng_rel_attention(qkv.data_ptr(), qkv.stride(0), q_col0, k_col0, v_col0, batch, heads, L,
                                   relbias.data_ptr(), kbias.data_ptr() if kbias is not None else None,
                                   out.data_ptr(), out.stride(0), split_off, stream_ptr()), "tng_rel_attention")


def cast_act(x, NB, H, W, y, *, Cc=None, upsample2x=False, act=ACT_NONE, act_param=0.0, split_off=0):
    require_cuda(x, y)
    Cc = x.shape[-1] if Cc is None else Cc
    n_out = NB * H * W * (4 if upsample2x else 1) * Cc
    _call("cast_act", NB * H * W * Cc * 4 + n_out * (4 if split_off else 2), load().tng_cast_act, x.data_ptr(), NB, H,
          W, Cc, x.stride(0), int(upsample2x), act, act_param, y.data_ptr(), y.stride(0), split_off, stream_ptr())


def softmax_rows(x, scale, y, *, L=None, split_off=0):
    require_cuda(x, y)
    rows = x.shape[0]
    L = x.shape[1] if L is None else L
    _call("softmax_rows", rows * L * (4 + (4 if split_off else 2)), load().tng_softmax_rows, x.data_ptr(), rows, L,
          x.stride(0), scale, y.data_ptr(), y.stride(0), split_off, stream_ptr())


def transpose_bf16(x, B, R, Cc, y):
    require_cuda(x, y)
    _call("transpose_bf16", B * R * Cc * 4, load().tng_transpose_bf16, x.data_ptr(), B, R, Cc, x.stride(0),
          y.data_ptr(), y.stride(0), stream_ptr())


def sched_step(model_out, cfg, guidance, sample, noise, coef, prev, next_in, *, B, Cc, HW, split_off=0):
    require_cuda(model_out, sample, noise, coef, prev, next_in)
    n = B * Cc * HW
    nbytes = n * 4 * ((2 if cfg else 1) * (model_out is not None) + 1 + (noise is not None) + (prev is not None)) \
        + (0 if next_in is None else n * (2 if cfg else 1) * (4 if split_off else 2))
    _call("sched_step", nbytes, load().tng_sched_step, ptr(model_out), 0 if model_out is None else model_out.stride(0),
          int(cfg), guidance, sample.data_ptr(), ptr(noise), coef.data_ptr(), ptr(prev), ptr(next_in),
          0 if next_in is None else next_in.stride(0), split_off, B, Cc, HW, stream_ptr())


def sched_multistep(model_out, cfg, guidance, sample, m1, m2, coef, order, m0, prev, next_in, *, B, Cc, HW,
                    split_off=0):
    """CFG combine + one multistep DPM-Solver update (coefficient row `coef`, see schedulers.py) + packing of the next
    UNet input. m1 / m2: the converted model outputs of the previous steps (read for order >= 2 / 3); m0 receives
    this step's."""
    require_cuda(model_out, sample, m1, m2, coef, m0, prev, next_in)
    n = B * Cc * HW
    reads = (2 if cfg else 1) + 1 + (order >= 2) + (order >= 3)
    nbytes = n * 4 * (reads + 1 + (prev is not None)) \
        + (0 if next_in is None else n * (2 if cfg else 1) * (4 if split_off else 2))
    _call("sched_multistep", nbytes, load().tng_sched_multistep, model_out.data_ptr(), model_out.stride(0), int(cfg),
          guidance, sample.data_ptr(), ptr(m1), ptr(m2), coef.data_ptr(), int(order), m0.data_ptr(), ptr(prev),
          ptr(next_in), 0 if next_in is None else next_in.stride(0), split_off, B, Cc, HW, stream_ptr())


def timestep_embedding(t, dim, flip_sin_to_cos, freq_shift, out):
    require_cuda(t, out)
    check(load().tng_timestep_embedding(t.data_ptr(), t.numel(), dim, int(flip_sin_to_cos), freq_shift,
                                        out.data_ptr(), stream_ptr()), "tng_timestep_embedding")


def linear_f32(x, w, b, y, *, pre_act=ACT_NONE, post_act=ACT_NONE):
    require_cuda(x, w, b, y)
    M, K = x.shape
    N = w.shape[0]
    check(load().tng_linear_f32(x.data_ptr(), M, K, w.data_ptr(), ptr(b), N, pre_act, post_act, y.data_ptr(),
                                stream_ptr()), "tng_linear_f32")


def convt_gather(Y, B, Lin, ktaps, Cout, stride, pad, Lout, bias, y):
    require_cuda(Y, bias, y)
    _call("convt_gather", (B * Lin * ktaps * Cout + B * Lout * Cout) * 4, load().tng_convt_gather, Y.data_ptr(), B, Lin,
          ktaps, Cout, stride, pad, Lout, ptr(bias), y.data_ptr(), stream_ptr())


def tanh_to_i16(x, n, ld_x, wave_f32, wave_i16):
    require_cuda(x, wave_f32, wave_i16)
    _call("tanh_to_i16", n * (4 + (4 if wave_f32 is not None else 0) + (2 if wave_i16 is not None else 0)),
          load().tng_tanh_to_i16, x.data_ptr(), n, ld_x, ptr(wave_f32), ptr(wave_i16), stream_ptr())


def stft_frames(y, pad, hi, lo):
    require_cuda(y, hi, lo)
    B, T = y.shape
    _call("stft_frames", B * T * 4 + 2 * hi.numel() * 2, load().tng_stft_frames, y.data_ptr(), B, T, pad, hi.data_ptr(),
          lo.data_ptr(), hi.stride(0), stream_ptr())


def stft_magnitude(F, bins, mag_op, split_off, log_mag, energy, floor=1e-5):
    require_cuda(F, mag_op, log_mag, energy)
    rows = F.shape[0]
    _call("stft_magnitude", rows * bins * (8 + 4 + 4), load().tng_stft_magnitude, F.data_ptr(), rows, bins, F.stride(0),
          ptr(mag_op), 0 if mag_op is None else mag_op.stride(0), split_off, ptr(log_mag), ptr(energy), floor,
          stream_ptr())


def log_clamp(x, y, floor=1e-5):
    require_cuda(x, y)
    _call("log_clamp", x.numel() * 8, load().tng_log_clamp, x.data_ptr(), x.numel(), floor, y.data_ptr(), stream_ptr())
