// HBM-bound glue kernels of the MetaPool / MetaConv variants (see include/avc_b200.h): GroupNorm statistics and
// apply, the pooling token mixer, patchify, LayerNorm + transpose, decoder-input assembly, code gathering.
// Every kernel reads fp32 channels-last tensors and writes the operand format of the consuming GEMM.
#include <cuda_bf16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_store.cuh"

namespace avc {

// ---------------------------------------------------------------- GroupNorm(1, C) statistics: one CTA per sample
__global__ void __launch_bounds__(512) gn_stats_kernel(const float* __restrict__ x, float* __restrict__ stats,
                                                       long long n, float eps) {
  const float4* xs = reinterpret_cast<const float4*>(x + (long long)blockIdx.x * n);
  double s = 0.0, ss = 0.0;
  for (long long i = threadIdx.x; i < n / 4; i += blockDim.x) {
    const float4 v = __ldg(xs + i);
    s += (double)v.x + (double)v.y + (double)v.z + (double)v.w;
    ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
  __shared__ double red[2][16];
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s;
    red[1][threadIdx.x >> 5] = ss;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) {
      a += red[0][i];
      b += red[1][i];
    }
    const double mean = a / (double)n;
    const double var = b / (double)n - mean * mean;      // biased variance
    stats[2 * blockIdx.x] = (float)mean;
    stats[2 * blockIdx.x + 1] = (float)(1.0 / sqrt(var + (double)eps));
  }
}

// ---------------------------------------------------------------- x + rstd*gamma_c*(avgpool3_t(x) - x)
__global__ void __launch_bounds__(256) gn_pool_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                                      const float* __restrict__ gamma, float* __restrict__ out_f32,
                                                      void* __restrict__ out_op, int mode, int round, long long total4,
                                                      int L, int C) {
  const int c4n = C >> 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;
    const int c = static_cast<int>(i - row * c4n) << 2;
    const long long b = row / L;
    const int t = static_cast<int>(row - b * L);
    const float rstd = __ldg(stats + 2 * b + 1);
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 xc = __ldg(reinterpret_cast<const float4*>(x + row * C + c));
    float4 sum = xc;
    float cnt = 1.0f;
    if (t > 0) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + (row - 1) * C + c));
      sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
      cnt += 1.0f;
    }
    if (t + 1 < L) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + (row + 1) * C + c));
      sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
      cnt += 1.0f;
    }
    const float inv = 1.0f / cnt;     // count_include_pad=False: edges average two samples
    float4 y;
    y.x = xc.x + rstd * g.x * (sum.x * inv - xc.x);
    y.y = xc.y + rstd * g.y * (sum.y * inv - xc.y);
    y.z = xc.z + rstd * g.z * (sum.z * inv - xc.z);
    y.w = xc.w + rstd * g.w * (sum.w * inv - xc.w);
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + row * C + c) = y;
    if (out_op) store_op4(out_op, mode, round, row, op_ld(C, mode), c, C, y);
  }
}

// ---------------------------------------------------------------- (x - mean)*rstd*gamma_c + beta_c
__global__ void __launch_bounds__(256) gn_apply_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       void* __restrict__ out_op, int mode, int round, long long total4,
                                                       int L, int C) {
  const int c4n = C >> 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;
    const int c = static_cast<int>(i - row * c4n) << 2;
    const long long b = row / L;
    const float mean = __ldg(stats + 2 * b), rstd = __ldg(stats + 2 * b + 1);
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 be = __ldg(reinterpret_cast<const float4*>(beta + c));
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + row * C + c));
    float4 y;
    y.x = (v.x - mean) * rstd * g.x + be.x;
    y.y = (v.y - mean) * rstd * g.y + be.y;
    y.z = (v.z - mean) * rstd * g.z + be.z;
    y.w = (v.w - mean) * rstd * g.w + be.w;
    store_op4(out_op, mode, round, row, op_ld(C, mode), c, C, y);
  }
}

// ---------------------------------------------------------------- batch-global mean / unbiased std (AdaIN "2" variants)
// x.mean(), x.std() over ALL elements of a tensor (factory/AutoVC2.py:60, factory/Norm.py:91-93).  Two deterministic
// stages: kGlobalParts CTAs write double partial sums in a fixed order, one CTA finishes.
constexpr int kGlobalParts = 256;

__global__ void __launch_bounds__(256) global_stats_partial_kernel(const float* __restrict__ x, long long n4,
                                                                   double* __restrict__ part) {
  const float4* xs = reinterpret_cast<const float4*>(x);
  double s = 0.0, ss = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(xs + i);
    s += (double)v.x + (double)v.y + (double)v.z + (double)v.w;
    ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
  __shared__ double red[2][8];
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s;
    red[1][threadIdx.x >> 5] = ss;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) {
      a += red[0][i];
      b += red[1][i];
    }
    part[2 * blockIdx.x] = a;
    part[2 * blockIdx.x + 1] = b;
  }
}

__global__ void global_stats_final_kernel(const double* __restrict__ part, int parts, long long n,
                                          float* __restrict__ stats) {
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < parts; ++i) {
      a += part[2 * i];
      b += part[2 * i + 1];
    }
    const double mean = a / (double)n;
    double var = (b - (double)n * mean * mean) / (double)(n - 1);      // torch.std(): Bessel-corrected
    if (var < 0.0) var = 0.0;
    stats[0] = (float)mean;
    stats[1] = (float)sqrt(var);
  }
}

// ---------------------------------------------------------------- AdaIN: (x - mean_x) / std_x * std_t + mu_t
__global__ void __launch_bounds__(256) adain_kernel(const float* __restrict__ x, const float* __restrict__ xs,
                                                    const float* __restrict__ ts, float* __restrict__ out_f32,
                                                    void* __restrict__ out_op, int mode, int round, long long total4,
                                                    int C) {
  const int c4n = C >> 2;
  const float mean = __ldg(xs), inv = 1.0f / __ldg(xs + 1), mu = __ldg(ts), sd = __ldg(ts + 1);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;
    const int c = static_cast<int>(i - row * c4n) << 2;
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + row * C + c));
    float4 y;      // same operation order as the reference: ((x - mean) / std) * std_t + mu_t
    y.x = (v.x - mean) * inv * sd + mu;
    y.y = (v.y - mean) * inv * sd + mu;
    y.z = (v.z - mean) * inv * sd + mu;
    y.w = (v.w - mean) * inv * sd + mu;
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + row * C + c) = y;
    if (out_op) store_op4(out_op, mode, round, row, op_ld(C, mode), c, C, y);
  }
}

// ---------------------------------------------------------------- patchify (+ GroupNorm(1, S))
// image I[h][w] = a[b][w][h] (h = channel, w = length).  token n = (h/p)*(S/p) + w/p, feature f = (h%p)*p + w%p.
// One thread per (w, h/4): reads 4 consecutive channels, writes 4 features p apart.
__global__ void __launch_bounds__(256) patchify_kernel(const float* __restrict__ a, const float* __restrict__ stats,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       void* __restrict__ out_op, int mode, int round, long long total4,
                                                       int S, int p) {
  const int c4n = S >> 2;
  const int npr = S / p;           // patches per image row
  const int F = p * p;
  const long long ld = op_ld(F, mode);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;                     // b*S + w
    const int h = static_cast<int>(i - row * c4n) << 2;
    const long long b = row / S;
    const int w = static_cast<int>(row - b * S);
    float4 v = __ldg(reinterpret_cast<const float4*>(a + row * S + h));
    if (stats) {
      const float mean = __ldg(stats + 2 * b), rstd = __ldg(stats + 2 * b + 1);
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + h));
      const float4 be = __ldg(reinterpret_cast<const float4*>(beta + h));
      v.x = (v.x - mean) * rstd * g.x + be.x;
      v.y = (v.y - mean) * rstd * g.y + be.y;
      v.z = (v.z - mean) * rstd * g.z + be.z;
      v.w = (v.w - mean) * rstd * g.w + be.w;
    }
    const float vals[4] = {v.x, v.y, v.z, v.w};
    const int wi = w / p, p2 = w - wi * p;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int hh = h + e;
      const int hi = hh / p, p1 = hh - hi * p;
      const long long tok = b * (long long)(npr * npr) + (long long)hi * npr + wi;
      store_op1(out_op, mode, round, tok, ld, p1 * p + p2, F, vals[e]);
    }
  }
}

// ---------------------------------------------------------------- LayerNorm statistics along rows / columns
// Moments as (count n, mean m, M2 = sum of squared deviations): Welford's update per element, Chan's formula to merge
// two partial sets.  The variance is never formed as E[x^2] - mean^2, which cancels in fp32 once |mean| is large next
// to the standard deviation (at |mean| / std = 1000 the normalised values were off by ~0.4); with centred sums the error
// grows only linearly in |mean| / std, with the length of the longest Welford chain plus the merge depth.
struct Moments {
  float n, m, M2;
};

// 1/n does not depend on the data, so it stays off the dependency chain through m; the approximate reciprocal (2 ulp)
// is well inside the error bound tests/test_gpu_meta_contract.py holds the statistics to
__device__ __forceinline__ void welford_add(Moments& a, float v) {
  a.n += 1.0f;
  const float inv_n = __fdividef(1.0f, a.n);
  const float d = v - a.m;
  a.m = fmaf(d, inv_n, a.m);
  a.M2 = fmaf(d, v - a.m, a.M2);
}

__device__ __forceinline__ Moments chan_merge(Moments a, Moments b) {
  const float n = a.n + b.n;
  if (n == 0.0f) return a;
  const float d = b.m - a.m, wb = __fdividef(b.n, n);
  return {n, fmaf(d, wb, a.m), a.M2 + b.M2 + d * d * (a.n * wb)};
}

// rows: one warp per row of C entries, lane l takes entries l, l + 32, ... (chains of ceil(C / 32)), then five merge
// levels across the warp.  Writes (mean, rstd) at stats[2 * row].
__global__ void __launch_bounds__(256) ln_row_stats_kernel(const float* __restrict__ x, float* __restrict__ stats,
                                                           long long rows, int C, float eps) {
  const long long row = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * C;
  Moments a = {0.f, 0.f, 0.f};
  for (int c = lane; c < C; c += 32) welford_add(a, __ldg(xr + c));
  for (int o = 16; o > 0; o >>= 1) {
    const Moments b = {__shfl_xor_sync(0xffffffffu, a.n, o), __shfl_xor_sync(0xffffffffu, a.m, o),
                       __shfl_xor_sync(0xffffffffu, a.M2, o)};
    a = chan_merge(a, b);
  }
  if (lane == 0) {
    stats[2 * row] = a.m;
    stats[2 * row + 1] = rsqrtf(a.M2 / C + eps);
  }
}

// cols: a block covers 32 columns x kColGroups row groups; thread (tx, ty) takes rows ty, ty + kColGroups, ... of
// column tx (a warp reads 32 consecutive floats of one row), then the groups merge in shared memory in a fixed tree
// (chains of ceil(R / kColGroups), three merge levels).  Writes (mean, rstd) at stats[2 * (b * C + c)].
constexpr int kColGroups = 8;
__global__ void __launch_bounds__(32 * kColGroups) ln_col_stats_kernel(const float* __restrict__ x,
                                                                       float* __restrict__ stats, int R, int C,
                                                                       float eps) {
  __shared__ Moments part[kColGroups][32];
  const int b = blockIdx.y, tx = threadIdx.x, ty = threadIdx.y;
  const int c = blockIdx.x * 32 + tx;
  Moments a = {0.f, 0.f, 0.f};
  if (c < C) {
    const float* xb = x + (long long)b * R * C + c;
    for (int r = ty; r < R; r += kColGroups) welford_add(a, __ldg(xb + (long long)r * C));
  }
  part[ty][tx] = a;
  for (int s = kColGroups / 2; s > 0; s >>= 1) {
    __syncthreads();
    if (ty < s) part[ty][tx] = chan_merge(part[ty][tx], part[ty + s][tx]);
  }
  if (ty == 0 && c < C) {
    const Moments t = part[0][tx];
    stats[2 * ((long long)b * C + c)] = t.m;
    stats[2 * ((long long)b * C + c) + 1] = rsqrtf(t.M2 / R + eps);
  }
}

// x [B][R][C] -> out [B][C][R_pad] (transposed), optional normalisation.  64 x 64 tiles through shared memory: the
// loads are float4 along C (a warp covers two 256-byte row segments), the stores are 8 consecutive r per thread --
// one 16-byte store per 16-bit operand row (two for the split format, two float4 for fp32 / the raw fp32 copy).
constexpr int kLnTile = 64;
__global__ void __launch_bounds__(256) ln_transpose_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, int ln_axis,
                                                           void* __restrict__ out_op, int mode, int round,
                                                           float* __restrict__ out_f32, int R, int C, int R_pad) {
  __shared__ float raw[kLnTile][kLnTile + 1];
  __shared__ float nrm[kLnTile][kLnTile + 1];
  const int b = blockIdx.z;
  const int r0 = blockIdx.y * kLnTile, c0 = blockIdx.x * kLnTile;
  const float* xb = x + (long long)b * R * C;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const bool vec = (C & 3) == 0;
#pragma unroll
  for (int i = 0; i < kLnTile / 16; ++i) {                 // coalesced along C
    const int lr = ty + 16 * i, r = r0 + lr, c = c0 + 4 * tx;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      if (vec && c + 3 < C) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(xb + (long long)r * C + c));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c + e < C) v[e] = __ldg(xb + (long long)r * C + c + e);
      }
    }
    // normalisation terms as (scale, shift) per element, fetched with 16-byte loads where the four columns are whole
    // (one scalar load per term and element made this pass issue 17 loads per float4 of data)
    float sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      if (ln_axis == 1) {
        const float2 st = __ldg(reinterpret_cast<const float2*>(stats + 2 * ((long long)b * R + r)));
        float g[4] = {0.f, 0.f, 0.f, 0.f}, be[4] = {0.f, 0.f, 0.f, 0.f};
        if (vec && c + 3 < C) {
          const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + c)), b4 = __ldg(reinterpret_cast<const float4*>(beta + c));
          g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w;
          be[0] = b4.x; be[1] = b4.y; be[2] = b4.z; be[3] = b4.w;
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (c + e < C) { g[e] = __ldg(gamma + c + e); be[e] = __ldg(beta + c + e); }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          sc[e] = st.y * g[e];
          sh[e] = be[e] - st.x * sc[e];
        }
      } else if (ln_axis == 2) {
        const float gr = __ldg(gamma + r), br = __ldg(beta + r);
        const float* st = stats + 2 * ((long long)b * C + c);
        float m[4] = {0.f, 0.f, 0.f, 0.f}, rs4[4] = {0.f, 0.f, 0.f, 0.f};
        if (vec && c + 3 < C) {      // (mean, rstd) pairs of four consecutive columns: 32 contiguous bytes, 16-byte aligned
          const float4 s0 = __ldg(reinterpret_cast<const float4*>(st)), s1 = __ldg(reinterpret_cast<const float4*>(st + 4));
          m[0] = s0.x; rs4[0] = s0.y; m[1] = s0.z; rs4[1] = s0.w; m[2] = s1.x; rs4[2] = s1.y; m[3] = s1.z; rs4[3] = s1.w;
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (c + e < C) { m[e] = st[2 * e]; rs4[e] = st[2 * e + 1]; }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          sc[e] = rs4[e] * gr;
          sh[e] = br - m[e] * sc[e];
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float n = v[e];
      if (ln_axis != 0 && r < R && c + e < C) n = fmaf(v[e], sc[e], sh[e]);
      raw[lr][4 * tx + e] = v[e];
      nrm[lr][4 * tx + e] = n;
    }
  }
  __syncthreads();
  const long long ld = op_ld(R_pad, mode);
  const int rg = threadIdx.x & 7;                          // group of 8 consecutive r (R_pad is a multiple of 8)
  const int r = r0 + 8 * rg;
  if (r >= R_pad) return;                                  // columns r in [R, R_pad) are written as zeros
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int lc = (threadIdx.x >> 3) + 32 * i, c = c0 + lc;
    if (c >= C) continue;
    const long long orow = (long long)b * C + c;
    float n[8], w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      n[j] = nrm[8 * rg + j][lc];
      w[j] = raw[8 * rg + j][lc];
    }
    if (out_op) {
      if (mode == 2) {
        float lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) lo[j] = n[j] - __bfloat162float(__float2bfloat16_rn(n[j]));
        __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out_op) + orow * ld + r;
        *reinterpret_cast<uint4*>(o) = make_uint4(pack_bf16(n[0], n[1]), pack_bf16(n[2], n[3]), pack_bf16(n[4], n[5]),
                                                  pack_bf16(n[6], n[7]));
        *reinterpret_cast<uint4*>(o + R_pad) = make_uint4(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]),
                                                          pack_bf16(lo[4], lo[5]), pack_bf16(lo[6], lo[7]));
      } else if (mode == 1) {
        *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out_op) + orow * ld + r) =
            make_uint4(pack_bf16(n[0], n[1]), pack_bf16(n[2], n[3]), pack_bf16(n[4], n[5]), pack_bf16(n[6], n[7]));
      } else if (mode == 3) {
        *reinterpret_cast<uint4*>(static_cast<__half*>(out_op) + orow * ld + r) =
            make_uint4(pack_f16(n[0], n[1]), pack_f16(n[2], n[3]), pack_f16(n[4], n[5]), pack_f16(n[6], n[7]));
      } else {
        float* o = static_cast<float*>(out_op) + orow * ld + r;
        if (round) {
#pragma unroll
          for (int j = 0; j < 8; ++j) n[j] = round_tf32(n[j]);
        }
        *reinterpret_cast<float4*>(o) = make_float4(n[0], n[1], n[2], n[3]);
        *reinterpret_cast<float4*>(o + 4) = make_float4(n[4], n[5], n[6], n[7]);
      }
    }
    if (out_f32) {
      float* o = out_f32 + orow * R_pad + r;
      *reinterpret_cast<float4*>(o) = make_float4(w[0], w[1], w[2], w[3]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(w[4], w[5], w[6], w[7]);
    }
  }
}

// ---------------------------------------------------------------- Meta decoder input / code gathering
__global__ void __launch_bounds__(256) meta_decoder_input_kernel(const float* __restrict__ codes,
                                                                 const float* __restrict__ c_trg,
                                                                 void* __restrict__ out_op, int mode, int round,
                                                                 long long total, int T, int freq, int H2, int E) {
  const int Fdim = H2 + E;
  const int n_codes = T / freq;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / T;                       // b*Fdim + f
    const int t = static_cast<int>(i - row * T);
    const long long b = row / Fdim;
    const int f = static_cast<int>(row - b * Fdim);
    const float v = f < H2 ? __ldg(codes + (b * n_codes + t / freq) * H2 + f) : __ldg(c_trg + b * E + (f - H2));
    store_op1(out_op, mode, round, row, op_ld(T, mode), t, T, v);
  }
}

__global__ void __launch_bounds__(256) gather_codes_kernel(const float* __restrict__ out, float* __restrict__ codes,
                                                           long long total, int T, int H, int freq) {
  const int n_codes = T / freq;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int u = static_cast<int>(i % (2 * H));
    const long long bj = i / (2 * H);
    const long long b = bj / n_codes;
    const int j = static_cast<int>(bj - b * n_codes);
    const int t = u < H ? j * freq + freq - 1 : j * freq;
    codes[i] = __ldg(out + (b * T + t) * (2LL * H) + u);
  }
}

static int grid_for(long long total, int block = 256) {
  long long blocks = (total + block - 1) / block;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace avc

using namespace avc;

extern "C" int avc_gn_stats(const float* x, float* stats, int B, long long n, float eps, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && stats && B > 0 && n > 0 && n % 4 == 0, "avc_gn_stats: bad arguments B=%d n=%lld", B, n);
  gn_stats_kernel<<<B, 512, 0, stream>>>(x, stats, n, eps);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_gn_pool_residual(const float* x, const float* stats, const float* gamma, float* out_f32,
                                    void* out_op, int out_dtype, int out_round_tf32, int B, int L, int C,
                                    void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && stats && gamma && (out_f32 || out_op), "avc_gn_pool_residual: null buffer");
  AVC_REQUIRE(B > 0 && L > 0 && C > 0 && C % 4 == 0 && out_dtype >= 0 && out_dtype <= 3, "avc_gn_pool_residual: bad shape");
  const long long total4 = (long long)B * L * (C / 4);
  gn_pool_kernel<<<grid_for(total4), 256, 0, stream>>>(x, stats, gamma, out_f32, out_op, out_dtype, out_round_tf32,
                                                       total4, L, C);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_gn_apply(const float* x, const float* stats, const float* gamma, const float* beta, void* out_op,
                            int out_dtype, int out_round_tf32, int B, int L, int C, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && stats && gamma && beta && out_op, "avc_gn_apply: null buffer");
  AVC_REQUIRE(B > 0 && L > 0 && C > 0 && C % 4 == 0 && out_dtype >= 0 && out_dtype <= 3, "avc_gn_apply: bad shape");
  const long long total4 = (long long)B * L * (C / 4);
  gn_apply_kernel<<<grid_for(total4), 256, 0, stream>>>(x, stats, gamma, beta, out_op, out_dtype, out_round_tf32,
                                                        total4, L, C);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_patchify(const float* a, const float* stats, const float* gamma, const float* beta, void* out_op,
                            int out_dtype, int out_round_tf32, int B, int S, int p, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(a && out_op, "avc_patchify: null buffer");
  AVC_REQUIRE(B > 0 && S > 0 && p > 0 && S % p == 0 && S % 4 == 0 && (p * p) % 8 == 0 && out_dtype >= 0 &&
                  out_dtype <= 3 && (!stats || (gamma && beta)),
              "avc_patchify: bad arguments S=%d p=%d", S, p);
  const long long total4 = (long long)B * S * (S / 4);
  patchify_kernel<<<grid_for(total4), 256, 0, stream>>>(a, stats, gamma, beta, out_op, out_dtype, out_round_tf32,
                                                        total4, S, p);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_ln_transpose(const float* x, const float* gamma, const float* beta, int ln_axis, void* out_op,
                                int out_dtype, int out_round_tf32, float* out_f32, float* scratch, int B, int R, int C,
                                void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && (out_op || out_f32), "avc_ln_transpose: null buffer");
  AVC_REQUIRE(B > 0 && B < 65536 && R > 0 && C > 0 && ln_axis >= 0 && ln_axis <= 2 && out_dtype >= 0 && out_dtype <= 3,
              "avc_ln_transpose: bad arguments");
  if (ln_axis) AVC_REQUIRE(gamma && beta && scratch, "avc_ln_transpose: LayerNorm needs gamma, beta and scratch");
  const int R_pad = (R + 7) / 8 * 8;
  if (ln_axis == 1) {
    const long long rows = (long long)B * R;
    ln_row_stats_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, stream>>>(x, scratch, rows, C, 1e-5f);
    count_launch();
  } else if (ln_axis == 2) {
    ln_col_stats_kernel<<<dim3((C + 31) / 32, B), dim3(32, kColGroups), 0, stream>>>(x, scratch, R, C, 1e-5f);
    count_launch();
  }
  dim3 grid((C + kLnTile - 1) / kLnTile, (R_pad + kLnTile - 1) / kLnTile, B);
  ln_transpose_kernel<<<grid, 256, 0, stream>>>(x, scratch, gamma, beta, ln_axis, out_op, out_dtype,
                                                         out_round_tf32, out_f32, R, C, R_pad);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_meta_decoder_input(const float* codes, const float* c_trg, void* out_op, int out_dtype,
                                      int out_round_tf32, int B, int T, int freq, int H2, int E, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(codes && c_trg && out_op, "avc_meta_decoder_input: null buffer");
  AVC_REQUIRE(B > 0 && T > 0 && freq > 0 && T % freq == 0 && T % 8 == 0 && H2 > 0 && E > 0 && out_dtype >= 0 &&
                  out_dtype <= 3,
              "avc_meta_decoder_input: bad shape");
  const long long total = (long long)B * (H2 + E) * T;
  meta_decoder_input_kernel<<<grid_for(total), 256, 0, stream>>>(codes, c_trg, out_op, out_dtype, out_round_tf32,
                                                                  total, T, freq, H2, E);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_gather_codes(const float* out, float* codes, int B, int T, int H, int freq, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(out && codes && B > 0 && T > 0 && H > 0 && freq > 0 && T % freq == 0, "avc_gather_codes: bad arguments");
  const long long total = (long long)B * (T / freq) * 2 * H;
  gather_codes_kernel<<<grid_for(total), 256, 0, stream>>>(out, codes, total, T, H, freq);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_global_stats(const float* x, long long n, float* stats, double* scratch, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && stats && scratch && n > 1 && n % 4 == 0, "avc_global_stats: bad arguments n=%lld", n);
  int parts = grid_for(n / 4);
  if (parts > kGlobalParts) parts = kGlobalParts;
  global_stats_partial_kernel<<<parts, 256, 0, stream>>>(x, n / 4, scratch);
  AVC_CHECK_CUDA(cudaGetLastError());
  global_stats_final_kernel<<<1, 32, 0, stream>>>(scratch, parts, n, stats);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch(2);
  return 0;
}

extern "C" int avc_adain(const float* x, const float* x_stats, const float* t_stats, float* out_f32, void* out_op,
                         int out_dtype, int out_round_tf32, long long rows, int C, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && x_stats && t_stats && (out_f32 || out_op), "avc_adain: null buffer");
  AVC_REQUIRE(rows > 0 && C > 0 && C % 4 == 0 && out_dtype >= 0 && out_dtype <= 3, "avc_adain: bad shape");
  const long long total4 = rows * (C / 4);
  adain_kernel<<<grid_for(total4), 256, 0, stream>>>(x, x_stats, t_stats, out_f32, out_op, out_dtype, out_round_tf32,
                                                     total4, C);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}
