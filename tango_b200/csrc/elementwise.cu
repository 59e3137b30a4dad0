// elementwise.cu — the HBM-bound kernels of the path: GroupNorm (two-source, +SiLU), LayerNorm, casts/upsample,
// row softmax, transpose, fused CFG + scheduler step, time embedding, ConvTranspose1d overlap-add, tanh->int16.
// All are coalesced / 16-byte vectorised along the contiguous channel dimension; statistics in fp32/fp64.
// See include/tango_b200.h for the reference call sites each entry point replaces.
#include "tng_ptx.cuh"
#include "tng_internal.h"

namespace tng {

__device__ __forceinline__ float4 load4(const void* base, int dt, long long idx) {
  if (dt == TNG_DT_F32) return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx);
  const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(base) + idx);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void store4_bf16(__nv_bfloat16* p, float4 v) {
  uint2 u;
  u.x = pack_bf16(v.x, v.y);
  u.y = pack_bf16(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ float bf16_lo(float v) { return v - __bfloat162float(__float2bfloat16_rn(v)); }
__device__ __forceinline__ void store4_split(__nv_bfloat16* p, float4 v, int split_off) {
  store4_bf16(p, v);
  if (split_off > 0) store4_bf16(p + split_off, make_float4(bf16_lo(v.x), bf16_lo(v.y), bf16_lo(v.z), bf16_lo(v.w)));
}
__device__ __forceinline__ float act_f(float x, int act, float p) {
  if (act == TNG_ACT_SILU) return silu_f(x);
  if (act == TNG_ACT_LRELU) return x > 0.f ? x : x * p;
  return x;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------------ GroupNorm
// Thread layout: a CTA owns GN_ROWS pixels of one image; thread t keeps a FIXED channel quad q = t % QT and walks the
// rows r = t / QT, + RL, ... (QT = min(C/4, 256) quad threads, RL = 256 / QT row lanes), so consecutive threads read
// consecutive 16-byte quads of a row (coalesced) and the per-channel constants live in registers.
constexpr int GN_ROWS_MAX = 128;  // pixels per CTA (upper bound; the host shrinks it for small grids)

template <bool BF>
__device__ __forceinline__ float4 ld_quad(const void* base, long long idx) {
  if (BF) {
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(base) + idx);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx);
}

template <bool BF>
__device__ __forceinline__ void gn_accum(const void* base, long long idx0, long long stride, int rl, int nrows, int RL,
                                         float* s, float* ss) {
  long long idx = idx0 + rl * stride;
  const long long step = RL * stride;
#pragma unroll 4
  for (int r = rl; r < nrows; r += RL, idx += step) {
    const float4 v = ld_quad<BF>(base, idx);
    s[0] += v.x; s[1] += v.y; s[2] += v.z; s[3] += v.w;
    ss[0] = fmaf(v.x, v.x, ss[0]); ss[1] = fmaf(v.y, v.y, ss[1]); ss[2] = fmaf(v.z, v.z, ss[2]); ss[3] = fmaf(v.w, v.w, ss[3]);
  }
}

// Per-(image, channel) sums and sums of squares (fp32 partials over this CTA's rows, fp64 atomics across CTAs).
__global__ void __launch_bounds__(256) col_stats_kernel(const void* x, int dt, int C, long long ld, long long HW,
                                                         double* stats, int GN_ROWS) {
  const int n = blockIdx.y;
  const long long r0 = static_cast<long long>(blockIdx.x) * GN_ROWS;
  const int Q = C / 4;
  const int QT = Q < 256 ? Q : 256;
  const int RL = 256 / QT;
  const int rl = threadIdx.x / QT;
  if (rl >= RL) return;
  const int nrows = static_cast<int>((HW - r0) < GN_ROWS ? (HW - r0) : GN_ROWS);
  for (int q = threadIdx.x - rl * QT; q < Q; q += QT) {
    const int c = q * 4;
    float s[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
    const long long idx0 = (n * HW + r0) * ld + c;
    if (dt == TNG_DT_F32) gn_accum<false>(x, idx0, ld, rl, nrows, RL, s, ss);
    else gn_accum<true>(x, idx0, ld, rl, nrows, RL, s, ss);
    double* sp = stats + (static_cast<long long>(n) * C + c) * 2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      atomicAdd(sp + 2 * j, static_cast<double>(s[j]));
      atomicAdd(sp + 2 * j + 1, static_cast<double>(ss[j]));
    }
  }
}

template <bool BF, bool SILU, bool SPLIT, bool RAW>
__device__ __forceinline__ void gn_apply_rows(const void* base, long long idx0, long long stride, int rl, int nrows, int RL,
                                              const float* sc, const float* sh, __nv_bfloat16* y, long long ystride,
                                              int split_off, __nv_bfloat16* raw, long long rstride, int raw_split_off) {
  // Rows rl, rl + RL, ... of this thread's 4 channels, in batches of UN: all loads of a batch are issued before the first
  // store (the compiler will not move a load above a store that may alias it, and one 16-byte load in flight per thread
  // leaves the kernel latency-bound), the last batch is predicated.
  constexpr int UN = 8;
  const int n = (nrows - rl + RL - 1) / RL;   // rows of this thread
  if (n <= 0) return;
  const int nb = (n + UN - 1) / UN;
  const int per = (n + nb - 1) / nb;          // balanced batches of at most UN rows
  long long idx = idx0 + rl * stride;
  const long long step = RL * stride;
  y += rl * ystride;
  const long long ystep = RL * ystride;
  if (RAW) raw += rl * rstride;
  const long long rstep = RL * rstride;
#pragma unroll 1
  for (int k0 = 0; k0 < n; k0 += per, idx += per * step, y += per * ystep) {
    const int cnt = (n - k0) < per ? (n - k0) : per;
    float4 v[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u)
      v[u] = (u < cnt) ? ld_quad<BF>(base, idx + u * step) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      if (u >= cnt) break;
      float4 o;
      o.x = fmaf(v[u].x, sc[0], sh[0]); o.y = fmaf(v[u].y, sc[1], sh[1]);
      o.z = fmaf(v[u].z, sc[2], sh[2]); o.w = fmaf(v[u].w, sc[3], sh[3]);
      if (SILU) { o.x = silu_f(o.x); o.y = silu_f(o.y); o.z = silu_f(o.z); o.w = silu_f(o.w); }
      __nv_bfloat16* yp = y + u * ystep;
      store4_bf16(yp, o);
      if (SPLIT) store4_bf16(yp + split_off, make_float4(bf16_lo(o.x), bf16_lo(o.y), bf16_lo(o.z), bf16_lo(o.w)));
      if (RAW) {
        __nv_bfloat16* rp = raw + u * rstep;
        store4_bf16(rp, v[u]);
        if (SPLIT) store4_bf16(rp + raw_split_off, make_float4(bf16_lo(v[u].x), bf16_lo(v[u].y), bf16_lo(v[u].z), bf16_lo(v[u].w)));
      }
    }
    if (RAW) raw += per * rstep;
  }
}

template <bool SILU, bool SPLIT, bool RAW>
__global__ void __launch_bounds__(256) gn_apply_kernel(const void* x0, int dt0, int C0, const double* stats0,
                                                        const void* x1, int dt1, int C1, const double* stats1,
                                                        long long HW, int groups, int tpg, int slab,
                                                        const float* gamma, const float* beta, float eps,
                                                        __nv_bfloat16* y, long long ld_y, int split_off,
                                                        __nv_bfloat16* raw, long long ld_raw, int raw_split_off, int GN_ROWS) {
  // A CTA owns GN_ROWS pixels of image blockIdx.y and the channel slab [c_lo, c_lo + slab) (whole groups, a multiple of
  // 4 channels): it reduces the per-channel accumulators of ITS groups only, so wide concatenated inputs (up to 2560
  // channels) do not make every CTA re-read the statistics of the whole tensor.
  __shared__ float s_mean[64], s_rstd[64];
  const int n = blockIdx.y;
  const int C = C0 + C1;
  const int cpg = C / groups;
  const int c_lo = blockIdx.z * slab;
  const int g_lo = c_lo / cpg, n_g = slab / cpg;
  {
    // tpg threads (a power of two <= 32, lanes of one warp) share a group
    const int gi = threadIdx.x / tpg, sub = threadIdx.x % tpg;
    const int g = g_lo + gi;
    double sum = 0.0, sq = 0.0;
    if (gi < n_g) {
      for (int c = g * cpg + sub; c < (g + 1) * cpg; c += tpg) {
        const double* sp = (c < C0) ? stats0 + (static_cast<long long>(n) * C0 + c) * 2
                                    : stats1 + (static_cast<long long>(n) * C1 + (c - C0)) * 2;
        sum += sp[0];
        sq += sp[1];
      }
    }
    for (int o = tpg >> 1; o > 0; o >>= 1) {
      sum += __shfl_xor_sync(0xffffffffu, sum, o);
      sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    if (gi < n_g && sub == 0) {
      const double cnt = static_cast<double>(HW) * cpg;
      const double mean = sum / cnt;
      double var = sq / cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      s_mean[gi] = static_cast<float>(mean);
      s_rstd[gi] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    }
  }
  __syncthreads();
  const long long r0 = static_cast<long long>(blockIdx.x) * GN_ROWS;
  const int nrows = static_cast<int>((HW - r0) < GN_ROWS ? (HW - r0) : GN_ROWS);
  const int Q = slab / 4;
  const int QT = Q < 256 ? Q : 256;
  const int RL = 256 / QT;
  const int rl = threadIdx.x / QT;
  if (rl >= RL) return;
  for (int q = threadIdx.x - rl * QT; q < Q; q += QT) {
    const int c = c_lo + q * 4;
    const bool first = c < C0;
    const void* base = first ? x0 : x1;
    const int dt = first ? dt0 : dt1;
    const int Cs = first ? C0 : C1;
    const int cc = first ? c : c - C0;
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(beta + c));
    float sc[4], sh[4];
    const float gm[4] = {g4.x, g4.y, g4.z, g4.w}, bt[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gi = (c + j) / cpg - g_lo;
      sc[j] = s_rstd[gi] * gm[j];
      sh[j] = bt[j] - s_mean[gi] * sc[j];
    }
    const long long rowb = n * HW + r0;
    __nv_bfloat16* yp = y + rowb * ld_y + c;
    __nv_bfloat16* rp = RAW ? raw + rowb * ld_raw + c : nullptr;
    if (dt == TNG_DT_F32)
      gn_apply_rows<false, SILU, SPLIT, RAW>(base, rowb * Cs + cc, Cs, rl, nrows, RL, sc, sh, yp, ld_y, split_off, rp, ld_raw, raw_split_off);
    else
      gn_apply_rows<true, SILU, SPLIT, RAW>(base, rowb * Cs + cc, Cs, rl, nrows, RL, sc, sh, yp, ld_y, split_off, rp, ld_raw, raw_split_off);
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// One warp per row, the row cached in registers (NI float4 per lane, C <= 128 * NI), so the variance is the exact
// two-pass form; NI is a template parameter so that no predicated-off iterations are issued. The grid is sized to the
// machine (a few CTAs per SM) and every warp walks rows with a stride, loading row r + stride while it normalises row
// r: the HBM latency of the next row hides behind the arithmetic and the stores of the current one.
template <int NI>
__device__ __forceinline__ void ln_load_row(const float* xr, int lane, int Q, float4* v) {
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int q = lane + i * 32;
    v[i] = (q < Q) ? *reinterpret_cast<const float4*>(xr + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

template <int NI, bool RMS>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* x, long long rows, int C, const float* gamma,
                                                         const float* beta, float eps, __nv_bfloat16* y, long long ld_y,
                                                         int split_off, float* yf) {
  const long long nwarps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int Q = C / 4;
  float4 v[NI], nx[NI];
  ln_load_row<NI>(x + row * C, lane, Q, v);
  for (; row < rows; row += nwarps) {
    const long long rn = row + nwarps;
    if (rn < rows) ln_load_row<NI>(x + rn * C, lane, Q, nx);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = RMS ? 0.f : warp_sum(s) / C;   // RMS (T5LayerNorm): no centring, no bias
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int q = lane + i * 32;
      if (q < Q) {
        const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        sq += a * a + b * b + c * c + d * d;
      }
    }
    const float rstd = rsqrtf(warp_sum(sq) / C + eps);
    __nv_bfloat16* yr = y + row * ld_y;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int q = lane + i * 32;
      if (q < Q) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + q * 4));
        const float4 b = RMS ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(reinterpret_cast<const float4*>(beta + q * 4));
        float4 o;
        o.x = (v[i].x - mean) * rstd * g.x + b.x;
        o.y = (v[i].y - mean) * rstd * g.y + b.y;
        o.z = (v[i].z - mean) * rstd * g.z + b.z;
        o.w = (v[i].w - mean) * rstd * g.w + b.w;
        if (y) store4_split(yr + q * 4, o, split_off);
        if (yf) *reinterpret_cast<float4*>(yf + row * C + q * 4) = o;   // optional fp32 copy (dense rows)
      }
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) v[i] = nx[i];
  }
}

// ------------------------------------------------------------------------------------------------ T5 front-end
// Embedding lookup: out[r, :] = table[ids[r], :] (fp32), one warp per row.
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* table, const long long* ids, long long rows, int C,
                                                           float* out) {
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* src = reinterpret_cast<const float4*>(table + ids[row] * C);
  float4* dst = reinterpret_cast<float4*>(out + row * C);
  for (int q = lane; q < C / 4; q += 32) dst[q] = __ldg(src + q);
}

// Self-attention with an additive (head, key - query) position bias and an additive per-key mask bias, no score
// scaling, head width 64 (T5Attention.forward of the `transformers` dependency): fp32 in, fp32 arithmetic, bf16 out.
// The sequences are short (<= 512 tokens), so this is a plain SIMT kernel: one CTA per (batch, head, 16 queries),
// each warp owns 4 queries; K / V stream through smem in 64-key tiles with an online softmax; lane j scores keys
// j and j + 32, lane d accumulates output dims d and d + 32.
constexpr int RA_KT = 64, RA_QPB = 16;
__global__ void __launch_bounds__(128) rel_attention_kernel(const float* qkv, long long ld, int q_col0, int k_col0,
                                                             int v_col0, int heads, int L, const float* relbias,
                                                             const float* kbias, __nv_bfloat16* out, long long ld_o,
                                                             int split_off) {
  __shared__ float sK[RA_KT][65];
  __shared__ float sV[RA_KT][65];
  __shared__ float sQ[4][64];
  __shared__ float sP[4][RA_KT];
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* base = qkv + static_cast<long long>(b) * L * ld + h * 64;
  const float* rb = relbias + static_cast<long long>(h) * (2 * L - 1) + (L - 1);   // rb[key - query]
  const float* kb = kbias ? kbias + static_cast<long long>(b) * L : nullptr;
  const int q_first = blockIdx.y * RA_QPB + warp * 4;
  float m[4], l[4], o0[4], o1[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { m[i] = -INFINITY; l[i] = 0.f; o0[i] = 0.f; o1[i] = 0.f; }
  for (int k0 = 0; k0 < L; k0 += RA_KT) {
    __syncthreads();   // previous tile fully consumed
    for (int e = threadIdx.x; e < RA_KT * 64; e += blockDim.x) {
      const int j = e >> 6, d = e & 63;
      const bool ok = (k0 + j) < L;
      sK[j][d] = ok ? base[static_cast<long long>(k0 + j) * ld + k_col0 + d] : 0.f;
      sV[j][d] = ok ? base[static_cast<long long>(k0 + j) * ld + v_col0 + d] : 0.f;
    }
    __syncthreads();
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
      const int q = q_first + i;
      if (q >= L) break;   // warp-uniform
      __syncwarp();
      sQ[warp][lane] = base[static_cast<long long>(q) * ld + q_col0 + lane];
      sQ[warp][lane + 32] = base[static_cast<long long>(q) * ld + q_col0 + lane + 32];
      __syncwarp();
      float s0 = 0.f, s1 = 0.f;
#pragma unroll 16
      for (int d = 0; d < 64; ++d) {
        const float qd = sQ[warp][d];
        s0 = fmaf(qd, sK[lane][d], s0);
        s1 = fmaf(qd, sK[lane + 32][d], s1);
      }
      const int j0 = k0 + lane, j1 = k0 + lane + 32;
      // scores += position_bias (relative bias + extended mask), as in T5Attention.forward
      s0 = (j0 < L) ? s0 + (rb[j0 - q] + (kb ? kb[j0] : 0.f)) : -INFINITY;
      s1 = (j1 < L) ? s1 + (rb[j1 - q] + (kb ? kb[j1] : 0.f)) : -INFINITY;
      const float m_new = fmaxf(m[i], warp_max(fmaxf(s0, s1)));
      const float corr = (m[i] == -INFINITY) ? 0.f : expf(m[i] - m_new);
      const float p0 = (j0 < L) ? expf(s0 - m_new) : 0.f;
      const float p1 = (j1 < L) ? expf(s1 - m_new) : 0.f;
      l[i] = l[i] * corr + warp_sum(p0 + p1);
      m[i] = m_new;
      sP[warp][lane] = p0;
      sP[warp][lane + 32] = p1;
      __syncwarp();
      float a0 = o0[i] * corr, a1 = o1[i] * corr;
#pragma unroll 16
      for (int j = 0; j < RA_KT; ++j) {
        const float pj = sP[warp][j];
        a0 = fmaf(pj, sV[j][lane], a0);
        a1 = fmaf(pj, sV[j][lane + 32], a1);
      }
      o0[i] = a0; o1[i] = a1;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = q_first + i;
    if (q >= L) break;
    const float inv = 1.0f / l[i];
    __nv_bfloat16* op = out + (static_cast<long long>(b) * L + q) * ld_o + h * 64;
    const float y0 = o0[i] * inv, y1 = o1[i] * inv;
    const __nv_bfloat16 h0 = __float2bfloat16_rn(y0), h1 = __float2bfloat16_rn(y1);
    op[lane] = h0;
    op[lane + 32] = h1;
    if (split_off > 0) {
      op[split_off + lane] = __float2bfloat16_rn(y0 - __bfloat162float(h0));
      op[split_off + lane + 32] = __float2bfloat16_rn(y1 - __bfloat162float(h1));
    }
  }
}

// ------------------------------------------------------------------------------------------------ cast / upsample
__global__ void __launch_bounds__(256) cast_act_kernel(const float* x, long long NB, int H, int W, int C, long long ld_x,
                                                        int up, int act, float act_param, __nv_bfloat16* y,
                                                        long long ld_y, int split_off) {
  const int Ho = up ? 2 * H : H, Wo = up ? 2 * W : W;
  const int Q = C / 4;
  const long long total = NB * Ho * Wo * Q;
  const long long gstride = static_cast<long long>(gridDim.x) * blockDim.x;
  constexpr int UN = 4;   // loads of UN grid-stride iterations are issued before the first store (see gn_apply_rows)
  for (long long i0 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i0 < total; i0 += UN * gstride) {
    float4 v[UN];
    long long oidx[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const long long i = i0 + u * gstride;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      oidx[u] = -1;
      if (i < total) {
        const int q = static_cast<int>(i % Q);
        const long long orow = i / Q;
        long long irow = orow;
        if (up) {
          const int wo = static_cast<int>(orow % Wo);
          const int ho = static_cast<int>((orow / Wo) % Ho);
          const long long n = orow / (static_cast<long long>(Wo) * Ho);
          irow = (n * H + (ho >> 1)) * W + (wo >> 1);
        }
        v[u] = *reinterpret_cast<const float4*>(x + irow * ld_x + q * 4);
        oidx[u] = orow * ld_y + q * 4;
      }
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      if (oidx[u] < 0) continue;
      float4 w = v[u];
      w.x = act_f(w.x, act, act_param); w.y = act_f(w.y, act, act_param);
      w.z = act_f(w.z, act, act_param); w.w = act_f(w.w, act, act_param);
      store4_split(y + oidx[u], w, split_off);
    }
  }
}

// ------------------------------------------------------------------------------------------------ row softmax
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* x, int L, long long ld_x, float scale,
                                                            __nv_bfloat16* y, long long ld_y, int split_off) {
  __shared__ float red[8];
  __shared__ float bc;
  const long long row = blockIdx.x;
  const float* xr = x + row * ld_x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float m = -INFINITY;
  for (int i = threadIdx.x; i < L; i += blockDim.x) m = fmaxf(m, xr[i] * scale);
  m = warp_max(m);
  if (lane == 0) red[warp] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = red[0];
    for (int i = 1; i < 8; ++i) t = fmaxf(t, red[i]);
    bc = t;
  }
  __syncthreads();
  m = bc;
  float s = 0.f;
  for (int i = threadIdx.x; i < L; i += blockDim.x) s += expf(xr[i] * scale - m);
  s = warp_sum(s);
  __syncthreads();
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    bc = t;
  }
  __syncthreads();
  const float inv = 1.0f / bc;
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    const float p = expf(xr[i] * scale - m) * inv;
    const __nv_bfloat16 hi = __float2bfloat16_rn(p);
    y[row * ld_y + i] = hi;
    if (split_off > 0) y[row * ld_y + split_off + i] = __float2bfloat16_rn(p - __bfloat162float(hi));
  }
}

// ------------------------------------------------------------------------------------------------ transpose
__global__ void __launch_bounds__(256) transpose_bf16_kernel(const __nv_bfloat16* x, int R, int C, long long ld_x,
                                                              __nv_bfloat16* y, long long ld_y) {
  __shared__ __nv_bfloat16 t[32][33];
  const long long b = blockIdx.z;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + tx;
    t[j][tx] = (r < R && c < C) ? x[(b * R + r) * ld_x + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + tx;
    if (c < C && r < R) y[(b * C + c) * ld_y + r] = t[tx][j];
  }
}

// ------------------------------------------------------------------------------------------------ CFG + scheduler
__global__ void __launch_bounds__(256) sched_step_kernel(const float* mo, long long ld_mo, int cfg, float guidance,
                                                          const float* sample, const float* noise, const float* coef,
                                                          float* prev, __nv_bfloat16* next_in, long long ld_in,
                                                          int split_off, long long B, int C, long long HW) {
  const float c_x0_s = coef[0], c_x0_m = coef[1], c_prev_x0 = coef[2], c_prev_s = coef[3], c_noise = coef[4];
  const float c_eps_s = coef[5], c_eps_m = coef[6], c_prev_eps = coef[7], clip = coef[8], c_x0_div = coef[9];
  const long long total = B * HW * C;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const long long hw = (i / C) % HW;
    const long long b = i / (C * HW);
    const long long nchw = (b * C + c) * HW + hw;
    const float s = sample[nchw];
    float out = s;
    if (mo) {
      float v;
      if (cfg) {
        const float u = mo[(b * HW + hw) * ld_mo + c];
        const float t = mo[((B + b) * HW + hw) * ld_mo + c];
        v = __fadd_rn(u, __fmul_rn(guidance, __fsub_rn(t, u)));  // models.py:246, no fma contraction
      } else {
        v = mo[(b * HW + hw) * ld_mo + c];
      }
      // scheduling_ddpm.py:306-311 / scheduling_ddim.py:303-313 with host-computed fp32 coefficients; the
      // multiplications and additions keep the reference's association order (no fma contraction).
      float x0 = __fdiv_rn(__fadd_rn(__fmul_rn(c_x0_s, s), __fmul_rn(c_x0_m, v)), c_x0_div);
      if (clip > 0.f) x0 = fminf(fmaxf(x0, -clip), clip);
      out = __fadd_rn(__fmul_rn(c_prev_x0, x0), __fmul_rn(c_prev_s, s));
      if (c_prev_eps != 0.f) {
        const float eps = __fadd_rn(__fmul_rn(c_eps_s, s), __fmul_rn(c_eps_m, v));
        out = __fadd_rn(out, __fmul_rn(c_prev_eps, eps));
      }
      if (noise && c_noise != 0.f) out = __fadd_rn(out, __fmul_rn(c_noise, noise[nchw]));
    }
    if (prev) prev[nchw] = out;
    if (next_in) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(out);
      const __nv_bfloat16 lo = __float2bfloat16_rn(out - __bfloat162float(hi));
      const long long r0 = (b * HW + hw) * ld_in + c;
      next_in[r0] = hi;
      if (split_off > 0) next_in[r0 + split_off] = lo;
      if (cfg) {
        const long long r1 = ((B + b) * HW + hw) * ld_in + c;
        next_in[r1] = hi;
        if (split_off > 0) next_in[r1 + split_off] = lo;
      }
    }
  }
}

// CFG + multistep DPM-Solver(++) update. coef = {c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4} (see
// include/tango_b200.h); m1 / m2 are read only when `order` needs them. Every product and sum is a separate
// round-to-nearest operation in the association order of scheduling_dpmsolver_multistep.py, so the result equals the
// fp32 CPU update bit for bit.
__global__ void __launch_bounds__(256) sched_multistep_kernel(const float* mo, long long ld_mo, int cfg, float guidance,
                                                               const float* sample, const float* m1, const float* m2,
                                                               const float* coef, int order, float* m0_out, float* prev,
                                                               __nv_bfloat16* next_in, long long ld_in, int split_off,
                                                               long long B, int C, long long HW) {
  const float c_s = coef[0], c_m = coef[1], c_div = coef[2], k_s = coef[3], k0 = coef[4], k1 = coef[5], k2 = coef[6];
  const float a1 = coef[7], a2 = coef[8], a3 = coef[9], a4 = coef[10];
  const long long total = B * HW * C;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const long long hw = (i / C) % HW;
    const long long b = i / (C * HW);
    const long long nchw = (b * C + c) * HW + hw;
    const float s = sample[nchw];
    float v;
    if (cfg) {
      const float u = mo[(b * HW + hw) * ld_mo + c];
      const float t = mo[((B + b) * HW + hw) * ld_mo + c];
      v = __fadd_rn(u, __fmul_rn(guidance, __fsub_rn(t, u)));
    } else {
      v = mo[(b * HW + hw) * ld_mo + c];
    }
    // convert_model_output: x0 (dpmsolver++) or eps (dpmsolver) for every prediction type
    const float m0 = __fdiv_rn(__fadd_rn(__fmul_rn(c_s, s), __fmul_rn(c_m, v)), c_div);
    float out = __fadd_rn(__fmul_rn(k_s, s), __fmul_rn(k0, m0));
    if (order == 2) {
      const float d1 = __fmul_rn(a1, __fsub_rn(m0, m1[nchw]));
      out = __fadd_rn(out, __fmul_rn(k1, d1));
    } else if (order == 3) {
      const float h1 = m1[nchw];
      const float e0 = __fmul_rn(a1, __fsub_rn(m0, h1));
      const float e1 = __fmul_rn(a2, __fsub_rn(h1, m2[nchw]));
      const float de = __fsub_rn(e0, e1);
      const float d1 = __fadd_rn(e0, __fmul_rn(a3, de));
      const float d2 = __fmul_rn(a4, de);
      out = __fadd_rn(__fadd_rn(out, __fmul_rn(k1, d1)), __fmul_rn(k2, d2));
    }
    m0_out[nchw] = m0;
    if (prev) prev[nchw] = out;
    if (next_in) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(out);
      const __nv_bfloat16 lo = __float2bfloat16_rn(out - __bfloat162float(hi));
      const long long r0 = (b * HW + hw) * ld_in + c;
      next_in[r0] = hi;
      if (split_off > 0) next_in[r0 + split_off] = lo;
      if (cfg) {
        const long long r1 = ((B + b) * HW + hw) * ld_in + c;
        next_in[r1] = hi;
        if (split_off > 0) next_in[r1 + split_off] = lo;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ time embedding
__global__ void timestep_embedding_kernel(const float* t, long long n, int dim, int flip, float freq_shift, float* out) {
  const int half = dim / 2;
  const long long total = n * half;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(i % half);
    const long long r = i / half;
    // embeddings.py:44-51: exponent = (-log(10000) * arange(half)) / (half - shift); emb = t * exp(exponent)
    const float exponent = __fdiv_rn(__fmul_rn(-9.210340371976184f, static_cast<float>(j)),
                                     static_cast<float>(half) - freq_shift);
    const float e = __fmul_rn(t[r], expf(exponent));
    const float sv = sinf(e), cv = cosf(e);
    float* o = out + r * dim;
    if (flip) { o[j] = cv; o[half + j] = sv; } else { o[j] = sv; o[half + j] = cv; }
    if ((dim & 1) && j == 0) o[dim - 1] = 0.f;
  }
}

// y[m, n] = post(sum_k pre(x[m,k]) * w[n,k] + b[n]); one warp per output element (tiny, exact fp32).
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* x, long long M, int K, const float* w,
                                                          const float* b, int N, int pre_act, int post_act, float* y) {
  const long long wid = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= M * N) return;
  const long long m = wid / N;
  const int n = static_cast<int>(wid % N);
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc += act_f(x[m * K + k], pre_act, 0.f) * w[static_cast<long long>(n) * K + k];
  acc = warp_sum(acc);
  if (lane == 0) y[m * N + n] = act_f(acc + (b ? b[n] : 0.f), post_act, 0.f);
}

// ------------------------------------------------------------------------------------------------ ConvTranspose1d
__global__ void __launch_bounds__(256) convt_gather_kernel(const float* Y, long long B, long long Lin, int ktaps, int Cout,
                                                            int stride, int pad, long long Lout, const float* bias,
                                                            float* y) {
  const int Q = Cout / 4;
  const long long total = B * Lout * Q;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int q = static_cast<int>(i % Q);
    const long long l = (i / Q) % Lout;
    const long long b = i / (Q * Lout);
    float4 acc = bias ? __ldg(reinterpret_cast<const float4*>(bias + q * 4)) : make_float4(0, 0, 0, 0);
    // l = qi*stride + t - pad  =>  t = l + pad - qi*stride in [0, ktaps)
    long long qi_hi = (l + pad) / stride;
    if (qi_hi > Lin - 1) qi_hi = Lin - 1;
    for (long long qi = qi_hi; qi >= 0; --qi) {
      const long long t = l + pad - qi * stride;
      if (t >= ktaps) break;
      const float4 v = *reinterpret_cast<const float4*>(Y + ((b * Lin + qi) * ktaps + t) * Cout + q * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(y + (b * Lout + l) * Cout + q * 4) = acc;
  }
}

__global__ void tanh_to_i16_kernel(const float* x, long long n, long long ld_x, float* wf, int16_t* wi) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float t = tanhf(x[i * ld_x]);
    if (wf) wf[i] = t;
    // hifigan/utilities.py:81: (wavs.cpu().numpy() * 32768).astype("int16") — float32 product, C cast toward
    // zero through int32 then wrap to int16 (tanh == 1.0 wraps to -32768, as in the reference).
    if (wi) wi[i] = static_cast<int16_t>(__float2int_rz(__fmul_rn(t, 32768.0f)));
  }
}

// ------------------------------------------------------------------------------------------------ STFT front-end
// y fp32 [B, T] -> reflect-padded (F.pad mode="reflect": no edge repeat) bf16 hi / lo planes [B, ld]; positions past
// T + 2*pad are zero. The frames of STFT.transform are then an OVERLAPPING strided view of these planes.
__global__ void __launch_bounds__(256) stft_frames_kernel(const float* y, long long B, long long T, int pad,
                                                           __nv_bfloat16* hi, __nv_bfloat16* lo, long long ld) {
  const long long total = B * ld;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / ld, j = i % ld;
    float v = 0.f;
    if (j < T + 2 * pad) {
      long long src = j - pad;
      if (src < 0) src = -src;
      else if (src >= T) src = 2 * (T - 1) - src;
      v = y[b * T + src];
    }
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

// One warp per frame: F [rows, ldF] = (real[0..bins) | imag[0..bins)) -> magnitude (bf16 hi/lo GEMM operand),
// log(max(mag, floor)) and the l2 norm over the bins (stft.py:74-77,178-184; audio_processing.py:85-91).
__global__ void __launch_bounds__(256) stft_magnitude_kernel(const float* F, long long rows, int bins, long long ldF,
                                                              __nv_bfloat16* op, long long ld_op, int split_off,
                                                              float* log_mag, float* energy, float floor_v) {
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* f = F + row * ldF;
  float e = 0.f;
  for (int b = lane; b < bins; b += 32) {
    const float re = f[b], im = f[bins + b];
    const float m = sqrtf(__fadd_rn(__fmul_rn(re, re), __fmul_rn(im, im)));
    e = fmaf(m, m, e);
    if (op) {
      const __nv_bfloat16 h = __float2bfloat16_rn(m);
      op[row * ld_op + b] = h;
      if (split_off > 0) op[row * ld_op + split_off + b] = __float2bfloat16_rn(m - __bfloat162float(h));
    }
    if (log_mag) log_mag[row * bins + b] = logf(fmaxf(m, floor_v));
  }
  e = warp_sum(e);
  if (energy && lane == 0) energy[row] = sqrtf(e);
}

__global__ void __launch_bounds__(256) log_clamp_kernel(const float* x, long long n, float floor_v, float* y) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    y[i] = logf(fmaxf(x[i], floor_v));
}

// pixels per GroupNorm CTA: enough CTAs (>= 4 per SM) even on the small-spatial levels
static inline int gn_rows_for(long long NB, long long HW) {
  long long rows = (NB * HW + 4LL * num_sms() - 1) / (4LL * num_sms());
  if (rows < 8) rows = 8;
  if (rows > GN_ROWS_MAX) rows = GN_ROWS_MAX;
  if (rows > HW) rows = HW;
  return static_cast<int>(rows);
}

// pixels per gn_apply CTA so that blocks * ceil(HW / rows) CTAs fit one wave of per_sm resident CTAs per SM
static inline int gn_rows_one_wave(long long blocks, long long HW, int per_sm) {
  long long gx = (static_cast<long long>(per_sm) * num_sms()) / (blocks > 0 ? blocks : 1);
  if (gx < 1) gx = 1;
  long long rows = (HW + gx - 1) / gx;
  if (rows < 8) rows = 8;
  if (rows > HW) rows = HW;
  return static_cast<int>(rows);
}

// LayerNorm grid: one warp per row up to 4 CTAs of `wpb` warps per SM, then the warps stride over the rows
static inline unsigned ln_grid(long long rows, int wpb) {
  long long g = (rows + wpb - 1) / wpb;
  const long long cap = 4LL * num_sms();
  if (g > cap) g = cap;
  return static_cast<unsigned>(g < 1 ? 1 : g);
}

static inline int grid_for(long long total, int block = 256) {
  long long g = (total + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace tng

using namespace tng;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

namespace tng {
int launch_col_stats(const void* x, int dt, long long C, long long ld, long long NB, long long HW, double* col_stats,
                     cudaStream_t st) {
  if (!x || !col_stats || C <= 0 || C % 4 || ld % 4 || NB <= 0 || HW <= 0 || (reinterpret_cast<uintptr_t>(x) & 7))
    return set_error(TNG_EINVAL, "groupnorm_stats: bad shape C=%lld ld=%lld", C, ld);
  const int gn_rows = gn_rows_for(NB, HW);
  dim3 grid((unsigned)((HW + gn_rows - 1) / gn_rows), (unsigned)NB);
  col_stats_kernel<<<grid, 256, 0, st>>>(x, dt, (int)C, ld, HW, col_stats, gn_rows);
  count_launch();
  return check_launch("col_stats");
}
}  // namespace tng

extern "C" int tng_groupnorm_stats(const void* x, int32_t dt, int64_t C, int64_t ld, int64_t NB, int64_t HW,
                                   double* col_stats, void* stream) {
  return launch_col_stats(x, dt, C, ld, NB, HW, col_stats, ST(stream));
}

extern "C" int tng_groupnorm_apply(const void* x0, int32_t dt0, int64_t C0, const double* stats0, const void* x1,
                                   int32_t dt1, int64_t C1, const double* stats1, int64_t NB, int64_t HW, int32_t groups,
                                   const float* gamma, const float* beta, float eps, int32_t act, void* y, int64_t ld_y,
                                   int32_t split_off, void* raw_bf16, int64_t ld_raw, int32_t raw_split_off, void* stream) {
  const int64_t C = C0 + (x1 ? C1 : 0);
  if (!x0 || !stats0 || (x1 && !stats1) || !y || groups <= 0 || groups > 64 || C % groups || C0 % 4 || (x1 && C1 % 4) ||
      ld_y % 4 || split_off % 4 || C > 8192)
    return set_error(TNG_EINVAL, "groupnorm_apply: bad shape");
  if (act != TNG_ACT_NONE && act != TNG_ACT_SILU) return set_error(TNG_EINVAL, "groupnorm_apply: act must be NONE or SILU");
  // channel slab per CTA: whole groups, a multiple of 4 channels, about 256-320 channels when the tensor is wider
  const int cpg = (int)(C / groups);
  int gps = 1;                                   // groups per slab
  while ((gps * cpg) % 4 != 0 && gps < groups) ++gps;
  while (gps * 2 * cpg <= 320 && groups % (gps * 2) == 0) gps *= 2;
  if ((gps * cpg) % 4 != 0 || groups % gps != 0) { gps = groups; }   // fall back: one slab = all channels
  const int slab = gps * cpg, nslabs = groups / gps;
  int tpg = 1;
  while (tpg * 2 * gps <= 256 && tpg < 32) tpg *= 2;
  const bool silu = act == TNG_ACT_SILU, split = split_off > 0, hasraw = raw_bf16 != nullptr;
  // One wave: the pixel blocks per (image, slab) are sized so that the grid fits the CTAs this instantiation can keep
  // resident (registers: 3 per SM for the plain variants), instead of leaving a partial second wave.
#define TNG_GN_LAUNCH(S, P, R)                                                                                           \
  do {                                                                                                                   \
    static int per_sm = 0;                                                                                               \
    if (per_sm == 0) {                                                                                                   \
      int v = 0;                                                                                                         \
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, gn_apply_kernel<S, P, R>, 256, 0) != cudaSuccess || v < 1)   \
        v = 2;                                                                                                           \
      per_sm = v;                                                                                                        \
    }                                                                                                                    \
    const int gn_rows = gn_rows_one_wave(NB * nslabs, HW, per_sm);                                                       \
    dim3 grid((unsigned)((HW + gn_rows - 1) / gn_rows), (unsigned)NB, (unsigned)nslabs);                                 \
    gn_apply_kernel<S, P, R><<<grid, 256, 0, ST(stream)>>>(x0, dt0, (int)C0, stats0, x1, dt1, x1 ? (int)C1 : 0, stats1,  \
                                                            HW, groups, tpg, slab, gamma, beta, eps,                     \
                                                            reinterpret_cast<__nv_bfloat16*>(y), ld_y, split_off,        \
                                                            reinterpret_cast<__nv_bfloat16*>(raw_bf16), ld_raw,          \
                                                            raw_split_off, gn_rows);                                     \
  } while (0)
  if (silu) {
    if (split) { if (hasraw) TNG_GN_LAUNCH(true, true, true); else TNG_GN_LAUNCH(true, true, false); }
    else { if (hasraw) TNG_GN_LAUNCH(true, false, true); else TNG_GN_LAUNCH(true, false, false); }
  } else {
    if (split) { if (hasraw) TNG_GN_LAUNCH(false, true, true); else TNG_GN_LAUNCH(false, true, false); }
    else { if (hasraw) TNG_GN_LAUNCH(false, false, true); else TNG_GN_LAUNCH(false, false, false); }
  }
#undef TNG_GN_LAUNCH
  count_launch();
  return check_launch("gn_apply");
}

extern "C" int tng_layernorm(const float* x, int64_t rows, int64_t C, const float* gamma, const float* beta, float eps,
                             void* y, int64_t ld_y, int32_t split_off, void* stream) {
  if (!x || !y || !gamma || !beta || C % 4 || C > 2048 || ld_y % 4 || split_off % 4) return set_error(TNG_EINVAL, "layernorm: C=%lld unsupported", (long long)C);
  const int wpb = 8;
  const unsigned grid = ln_grid(rows, wpb);
  const int ni = (int)((C / 4 + 31) / 32);
#define TNG_LN(NI) layernorm_kernel<NI, false><<<grid, wpb * 32, 0, ST(stream)>>>(x, rows, (int)C, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(y), ld_y, split_off, nullptr)
  if (ni <= 1) TNG_LN(1);
  else if (ni <= 2) TNG_LN(2);
  else if (ni <= 3) TNG_LN(3);
  else if (ni <= 5) TNG_LN(5);
  else if (ni <= 10) TNG_LN(10);
  else TNG_LN(16);
#undef TNG_LN
  count_launch();
  return check_launch("layernorm");
}

extern "C" int tng_rmsnorm(const float* x, int64_t rows, int64_t C, const float* gamma, float eps, void* y, int64_t ld_y,
                           int32_t split_off, float* y_f32, void* stream) {
  if (!x || (!y && !y_f32) || !gamma || C % 4 || C > 2048 || ld_y % 4 || split_off % 4) return set_error(TNG_EINVAL, "rmsnorm: C=%lld unsupported", (long long)C);
  const int wpb = 8;
  const unsigned grid = ln_grid(rows, wpb);
  const int ni = (int)((C / 4 + 31) / 32);
  const float* beta = nullptr;
#define TNG_RMS(NI) layernorm_kernel<NI, true><<<grid, wpb * 32, 0, ST(stream)>>>(x, rows, (int)C, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(y), ld_y, split_off, y_f32)
  if (ni <= 1) TNG_RMS(1);
  else if (ni <= 2) TNG_RMS(2);
  else if (ni <= 3) TNG_RMS(3);
  else if (ni <= 5) TNG_RMS(5);
  else if (ni <= 10) TNG_RMS(10);
  else TNG_RMS(16);
#undef TNG_RMS
  count_launch();
  return check_launch("rmsnorm");
}

extern "C" int tng_gather_rows(const float* table, int64_t n_table_rows, const int64_t* ids, int64_t rows, int64_t C,
                               float* out, void* stream) {
  if (!table || !ids || !out || rows <= 0 || n_table_rows <= 0 || C % 4 ||
      ((reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(out)) & 15))
    return set_error(TNG_EINVAL, "gather_rows: bad argument");
  const int wpb = 8;
  gather_rows_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, ST(stream)>>>(
      table, reinterpret_cast<const long long*>(ids), rows, (int)C, out);
  count_launch();
  return check_launch("gather_rows");
}

extern "C" int tng_rel_attention(const float* qkv, int64_t ld, int32_t q_col0, int32_t k_col0, int32_t v_col0,
                                 int32_t batch, int32_t heads, int32_t L, const float* relbias, const float* kbias,
                                 void* out, int64_t ld_o, int32_t split_off, void* stream) {
  if (!qkv || !relbias || !out || batch <= 0 || heads <= 0 || L <= 0) return set_error(TNG_EINVAL, "rel_attention: bad argument");
  dim3 grid((unsigned)(batch * heads), (unsigned)((L + RA_QPB - 1) / RA_QPB));
  rel_attention_kernel<<<grid, 128, 0, ST(stream)>>>(qkv, ld, q_col0, k_col0, v_col0, heads, L, relbias, kbias,
                                                      reinterpret_cast<__nv_bfloat16*>(out), ld_o, split_off);
  count_launch();
  return check_launch("rel_attention");
}

extern "C" int tng_cast_act(const float* x, int64_t NB, int64_t H, int64_t W, int64_t C, int64_t ld_x,
                            int32_t upsample2x, int32_t act, float act_param, void* y, int64_t ld_y, int32_t split_off,
                            void* stream) {
  if (!x || !y || C % 4 || ld_x % 4 || ld_y % 4 || split_off % 4) return set_error(TNG_EINVAL, "cast_act: bad shape");
  const long long total = NB * H * W * (upsample2x ? 4 : 1) * (C / 4);
  cast_act_kernel<<<grid_for(total), 256, 0, ST(stream)>>>(x, NB, (int)H, (int)W, (int)C, ld_x, upsample2x, act, act_param,
                                                            reinterpret_cast<__nv_bfloat16*>(y), ld_y, split_off);
  count_launch();
  return check_launch("cast_act");
}

extern "C" int tng_softmax_rows(const float* x, int64_t rows, int64_t L, int64_t ld_x, float scale, void* y,
                                int64_t ld_y, int32_t split_off, void* stream) {
  if (!x || !y || rows <= 0 || L <= 0) return set_error(TNG_EINVAL, "softmax_rows: bad shape");
  softmax_rows_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(x, (int)L, ld_x, scale, reinterpret_cast<__nv_bfloat16*>(y),
                                                               ld_y, split_off);
  count_launch();
  return check_launch("softmax_rows");
}

extern "C" int tng_transpose_bf16(const void* x, int64_t B, int64_t R, int64_t C, int64_t ld_x, void* y, int64_t ld_y,
                                  void* stream) {
  if (!x || !y) return set_error(TNG_EINVAL, "transpose: null");
  dim3 grid((unsigned)((C + 31) / 32), (unsigned)((R + 31) / 32), (unsigned)B);
  transpose_bf16_kernel<<<grid, 256, 0, ST(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), (int)R, (int)C, ld_x,
                                                       reinterpret_cast<__nv_bfloat16*>(y), ld_y);
  count_launch();
  return check_launch("transpose");
}

extern "C" int tng_sched_step(const float* model_out, int64_t ld_mo, int32_t cfg, float guidance, const float* sample,
                              const float* noise, const float* coef, float* prev, void* next_in, int64_t ld_in,
                              int32_t split_off, int64_t B, int64_t C, int64_t HW, void* stream) {
  if (!sample || !coef || (!prev && !next_in)) return set_error(TNG_EINVAL, "sched_step: null argument");
  sched_step_kernel<<<grid_for(B * C * HW), 256, 0, ST(stream)>>>(model_out, ld_mo, cfg, guidance, sample, noise, coef, prev,
                                                                  reinterpret_cast<__nv_bfloat16*>(next_in), ld_in,
                                                                  split_off, B, (int)C, HW);
  count_launch();
  return check_launch("sched_step");
}

extern "C" int tng_sched_multistep(const float* model_out, int64_t ld_mo, int32_t cfg, float guidance,
                                   const float* sample, const float* m1, const float* m2, const float* coef,
                                   int32_t order, float* m0, float* prev, void* next_in, int64_t ld_in,
                                   int32_t split_off, int64_t B, int64_t C, int64_t HW, void* stream) {
  if (!model_out || !sample || !coef || !m0 || (!prev && !next_in))
    return set_error(TNG_EINVAL, "sched_multistep: null argument");
  if (order < 1 || order > 3) return set_error(TNG_EINVAL, "sched_multistep: order %d not in {1, 2, 3}", (int)order);
  if ((order >= 2 && !m1) || (order == 3 && !m2))
    return set_error(TNG_EINVAL, "sched_multistep: order %d needs %s", (int)order, order == 2 ? "m1" : "m1 and m2");
  if (B <= 0 || C <= 0 || HW <= 0 || ld_mo < C || split_off < 0 || (next_in && ld_in < C + split_off))
    return set_error(TNG_EINVAL, "sched_multistep: bad shape (B=%lld C=%lld HW=%lld ld_mo=%lld ld_in=%lld split_off=%d)",
                     (long long)B, (long long)C, (long long)HW, (long long)ld_mo, (long long)ld_in, (int)split_off);
  if (m0 == m1 || m0 == m2 || m0 == sample || (order == 3 && m1 == m2))
    return set_error(TNG_EINVAL, "sched_multistep: m0 / m1 / m2 / sample must be distinct buffers");
  sched_multistep_kernel<<<grid_for(B * C * HW), 256, 0, ST(stream)>>>(
      model_out, ld_mo, cfg, guidance, sample, m1, m2, coef, order, m0, prev, reinterpret_cast<__nv_bfloat16*>(next_in),
      ld_in, split_off, B, (int)C, HW);
  count_launch();
  return check_launch("sched_multistep");
}

extern "C" int tng_timestep_embedding(const float* t, int64_t n, int32_t dim, int32_t flip_sin_to_cos, float freq_shift,
                                      float* out, void* stream) {
  if (!t || !out || dim < 2) return set_error(TNG_EINVAL, "timestep_embedding: bad argument");
  timestep_embedding_kernel<<<grid_for(n * (dim / 2)), 256, 0, ST(stream)>>>(t, n, dim, flip_sin_to_cos, freq_shift, out);
  count_launch();
  return check_launch("timestep_embedding");
}

extern "C" int tng_linear_f32(const float* x, int64_t M, int64_t K, const float* w, const float* b, int64_t N,
                              int32_t pre_act, int32_t post_act, float* y, void* stream) {
  if (!x || !w || !y) return set_error(TNG_EINVAL, "linear_f32: null");
  const long long threads = M * N * 32;
  linear_f32_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ST(stream)>>>(x, M, (int)K, w, b, (int)N, pre_act, post_act, y);
  count_launch();
  return check_launch("linear_f32");
}

extern "C" int tng_convt_gather(const float* Y, int64_t B, int64_t Lin, int32_t ktaps, int64_t Cout, int32_t stride,
                                int32_t pad, int64_t Lout, const float* bias, float* y, void* stream) {
  if (!Y || !y || Cout % 4) return set_error(TNG_EINVAL, "convt_gather: bad shape");
  convt_gather_kernel<<<grid_for(B * Lout * (Cout / 4)), 256, 0, ST(stream)>>>(Y, B, Lin, ktaps, (int)Cout, stride, pad, Lout,
                                                                               bias, y);
  count_launch();
  return check_launch("convt_gather");
}

extern "C" int tng_tanh_to_i16(const float* x, int64_t n, int64_t ld_x, float* wave_f32, int16_t* wave_i16, void* stream) {
  if (!x) return set_error(TNG_EINVAL, "tanh_to_i16: null");
  tanh_to_i16_kernel<<<grid_for(n), 256, 0, ST(stream)>>>(x, n, ld_x, wave_f32, wave_i16);
  count_launch();
  return check_launch("tanh_to_i16");
}

extern "C" int tng_stft_frames(const float* y, int64_t B, int64_t T, int32_t pad, void* hi, void* lo, int64_t ld,
                               void* stream) {
  if (!y || !hi || !lo || B <= 0 || T <= pad || pad < 0 || ld < T + 2 * pad)
    return set_error(TNG_EINVAL, "stft_frames: bad argument (reflect padding needs T > pad)");
  stft_frames_kernel<<<grid_for(B * ld), 256, 0, ST(stream)>>>(y, B, T, pad, reinterpret_cast<__nv_bfloat16*>(hi),
                                                                reinterpret_cast<__nv_bfloat16*>(lo), ld);
  count_launch();
  return check_launch("stft_frames");
}

extern "C" int tng_stft_magnitude(const float* F, int64_t rows, int32_t bins, int64_t ldF, void* mag_op, int64_t ld_op,
                                  int32_t split_off, float* log_mag, float* energy, float floor_v, void* stream) {
  if (!F || rows <= 0 || bins <= 0 || ldF < 2 * bins) return set_error(TNG_EINVAL, "stft_magnitude: bad argument");
  const int wpb = 8;
  stft_magnitude_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, ST(stream)>>>(
      F, rows, bins, ldF, reinterpret_cast<__nv_bfloat16*>(mag_op), ld_op, split_off, log_mag, energy, floor_v);
  count_launch();
  return check_launch("stft_magnitude");
}

extern "C" int tng_log_clamp(const float* x, int64_t n, float floor_v, float* y, void* stream) {
  if (!x || !y || n <= 0) return set_error(TNG_EINVAL, "log_clamp: bad argument");
  log_clamp_kernel<<<grid_for(n), 256, 0, ST(stream)>>>(x, n, floor_v, y);
  count_launch();
  return check_launch("log_clamp");
}
