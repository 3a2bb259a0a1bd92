// Batch-statistics BatchNorm (nn.BatchNorm1d in training mode) for the conv + BN layers: the per-channel batch
// reduction with the running-buffer update, and the normalise / activate / store pass (see include/avc_b200.h).
// Both are HBM-bound streaming passes over the conv output v [rows][ld] fp32: float4 loads along the channels, so a
// warp reads 512 contiguous bytes of one row.
#include <cuda_bf16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_store.cuh"

namespace avc {

constexpr int kBnCols4 = 32;                 // float4 columns per CTA (128 channels, one per lane)
constexpr int kBnRowLanes = 8;               // row lanes per CTA: 256 threads
constexpr int kBnThreads = kBnCols4 * kBnRowLanes;
constexpr int kBnHeader = 2;                 // doubles in front of the partials: num_batches_tracked snapshot + pad

// ---------------------------------------------------------------- stage 1: fp64 partial sums per (row chunk, channel)
// CTA (x, y) sums rows [y * rows_per_part, +rows_per_part) of channels [128 x, +128).  Row lane ty takes rows ty,
// ty + 8, ... in order; the eight lanes are then added in lane order.  Fixed order throughout: bitwise deterministic.
__global__ void __launch_bounds__(kBnThreads) bn_stats_partial_kernel(const float* __restrict__ v, long long rows,
                                                                     int C, long long ld, long long rows_per_part,
                                                                     double* __restrict__ scratch,
                                                                     const long long* __restrict__ nbt) {
  const int tx = threadIdx.x & (kBnCols4 - 1), ty = threadIdx.x / kBnCols4;
  const int c = (blockIdx.x * kBnCols4 + tx) * 4;
  const long long r0 = blockIdx.y * rows_per_part;
  const long long r1 = min(rows, r0 + rows_per_part);
  double s[4] = {0.0, 0.0, 0.0, 0.0}, ss[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < C) {
    const float* p = v + c;
    long long r = r0 + ty;
    // four rows in flight per thread
    for (; r + 3 * kBnRowLanes < r1; r += 4 * kBnRowLanes) {
      float4 q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) q[u] = __ldg(reinterpret_cast<const float4*>(p + (r + u * kBnRowLanes) * ld));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double x0 = q[u].x, x1 = q[u].y, x2 = q[u].z, x3 = q[u].w;
        s[0] += x0; s[1] += x1; s[2] += x2; s[3] += x3;
        ss[0] = fma(x0, x0, ss[0]); ss[1] = fma(x1, x1, ss[1]); ss[2] = fma(x2, x2, ss[2]); ss[3] = fma(x3, x3, ss[3]);
      }
    }
    for (; r < r1; r += kBnRowLanes) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(p + r * ld));
      const double x0 = q.x, x1 = q.y, x2 = q.z, x3 = q.w;
      s[0] += x0; s[1] += x1; s[2] += x2; s[3] += x3;
      ss[0] = fma(x0, x0, ss[0]); ss[1] = fma(x1, x1, ss[1]); ss[2] = fma(x2, x2, ss[2]); ss[3] = fma(x3, x3, ss[3]);
    }
  }
  __shared__ double red[2][kBnRowLanes][kBnCols4 * 4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    red[0][ty][4 * tx + e] = s[e];
    red[1][ty][4 * tx + e] = ss[e];
  }
  __syncthreads();
  // 256 threads write the 2 x 128 sums of this CTA: thread i -> (sum kind i / 128, channel i % 128)
  const int kind = threadIdx.x >> 7, cl = threadIdx.x & 127;
  const int ch = blockIdx.x * kBnCols4 * 4 + cl;
  if (ch < C) {
    double a = 0.0;
#pragma unroll
    for (int i = 0; i < kBnRowLanes; ++i) a += red[kind][i][cl];
    scratch[kBnHeader + (2LL * blockIdx.y + kind) * C + ch] = a;
  }
  if (nbt && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0)
    reinterpret_cast<long long*>(scratch)[0] = *nbt;      // snapshot: stage 2 reads it, then overwrites the buffer
}

// ---------------------------------------------------------------- stage 2: merge, scale / shift, running buffers
// CTA x owns channels [32 x, +32); its eight warps add parts w, w + 8, ... in order, then the warps' sums are added in
// warp order.  Every CTA reads the count from the snapshot stage 1 took, so CTA 0 may overwrite num_batches_tracked.
__global__ void __launch_bounds__(kBnThreads) bn_stats_final_kernel(const double* __restrict__ scratch, int parts,
                                                                   long long rows, int C, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, float eps,
                                                                   float momentum, int cumulative,
                                                                   float* __restrict__ running_mean,
                                                                   float* __restrict__ running_var,
                                                                   long long* __restrict__ nbt,
                                                                   float* __restrict__ scale_shift) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const double* part = scratch + kBnHeader;
  double s = 0.0, ss = 0.0;
  if (c < C) {
    for (int p = w; p < parts; p += kBnRowLanes) {
      s += part[2LL * p * C + c];
      ss += part[(2LL * p + 1) * C + c];
    }
  }
  __shared__ double red[2][kBnRowLanes][32];
  red[0][w][lane] = s;
  red[1][w][lane] = ss;
  __syncthreads();
  const long long count = nbt ? reinterpret_cast<const long long*>(scratch)[0] + 1 : 0;
  if (w == 0 && c < C) {
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int i = 0; i < kBnRowLanes; ++i) {
      a += red[0][i][lane];
      b += red[1][i][lane];
    }
    const double n = (double)rows;
    const double mean = a / n;
    double var = b / n - mean * mean;                      // biased: what the batch is normalised with
    if (var < 0.0) var = 0.0;
    const double scale = (double)gamma[c] / sqrt(var + (double)eps);
    scale_shift[c] = (float)scale;
    scale_shift[C + c] = (float)((double)beta[c] - mean * scale);
    if (running_mean) {
      const double m = cumulative ? 1.0 / (double)count : (double)momentum;
      running_mean[c] = (float)((1.0 - m) * (double)running_mean[c] + m * mean);
      running_var[c] = (float)((1.0 - m) * (double)running_var[c] + m * var * (n / (n - 1.0)));   // unbiased
    }
  }
  if (nbt && blockIdx.x == 0 && threadIdx.x == 0) *nbt = count;
}

// ---------------------------------------------------------------- act(scale * v + shift) (+ residual) -> out / out2
// Thread (tx, ty) of CTA (x, y) keeps the scale / shift of its four channels in registers and walks rows
// y * 8 + ty, stepping 8 * gridDim.y.
__device__ __forceinline__ float bn_act(int act, float y) {
  if (act == AVC_ACT_RELU) return fmaxf(y, 0.0f);
  if (act == AVC_ACT_TANH) return tanh_fast(y);            // the GEMM epilogue's tanh (avc_gemm.cu apply_act)
  return y;
}

__global__ void __launch_bounds__(kBnThreads) bn_apply_kernel(avc_bn_apply_desc d) {
  const int tx = threadIdx.x & (kBnCols4 - 1), ty = threadIdx.x / kBnCols4;
  const int C = d.C;
  const int c = (blockIdx.x * kBnCols4 + tx) * 4;
  if (c >= C) return;
  const float4 sc = __ldg(reinterpret_cast<const float4*>(d.scale_shift + c));
  const float4 sh = __ldg(reinterpret_cast<const float4*>(d.scale_shift + C + c));
  const float* __restrict__ v = d.v;
  const float* __restrict__ res = d.residual;
  const int rows = d.B * d.T;
  const int step = kBnRowLanes * gridDim.y;
#pragma unroll 2
  for (int r = blockIdx.y * kBnRowLanes + ty; r < rows; r += step) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(v + r * d.v_ld + c));
    float y[4] = {fmaf(sc.x, x.x, sh.x), fmaf(sc.y, x.y, sh.y), fmaf(sc.z, x.z, sh.z), fmaf(sc.w, x.w, sh.w)};
    float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (res) {
      rv = __ldg(reinterpret_cast<const float4*>(res + r * d.res_ld + c));
      if (!d.res_after_act) { y[0] += rv.x; y[1] += rv.y; y[2] += rv.z; y[3] += rv.w; }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) y[e] = bn_act(d.act, y[e]);
    if (res && d.res_after_act) { y[0] += rv.x; y[1] += rv.y; y[2] += rv.z; y[3] += rv.w; }
    const float4 o = make_float4(y[0], y[1], y[2], y[3]);
    if (d.out2) *reinterpret_cast<float4*>(d.out2 + r * d.out2_ld + c) = o;
    if (d.out) {
      const int b = r / d.T, t = r - b * d.T;
      store_op4(d.out, d.out_dtype, d.out_round_tf32, (long long)b * d.out_rows_per_utt + d.out_row0 + t, d.out_ld, c, C,
                o);
    }
  }
}

static int bn_parts(long long rows, int gx) {
  long long parts = (4LL * num_sms() + gx - 1) / gx;       // about four CTAs per SM
  const long long by_rows = (rows + 31) / 32;              // at least 32 rows per part
  if (parts > by_rows) parts = by_rows;
  if (parts > AVC_BN_MAX_PARTS) parts = AVC_BN_MAX_PARTS;
  return parts < 1 ? 1 : (int)parts;
}

}  // namespace avc

using namespace avc;

extern "C" int avc_bn_batch_stats(const float* v, long long rows, int C, long long v_ld, const float* gamma,
                                  const float* beta, float eps, float momentum, int cumulative, float* running_mean,
                                  float* running_var, long long* num_batches_tracked, float* scale_shift,
                                  double* scratch, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(v && gamma && beta && scale_shift && scratch, "avc_bn_batch_stats: null buffer");
  AVC_REQUIRE(rows > 1 && C > 0 && C % 4 == 0 && v_ld >= C && v_ld % 4 == 0 && eps > 0.0f,
              "avc_bn_batch_stats: bad shape rows=%lld C=%d ld=%lld (need rows > 1, C %% 4 == 0)", rows, C, v_ld);
  AVC_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "avc_bn_batch_stats: running_mean / running_var");
  AVC_REQUIRE(!cumulative || (num_batches_tracked && running_mean),
              "avc_bn_batch_stats: the cumulative average needs num_batches_tracked and the running buffers");
  const int gx = (C / 4 + kBnCols4 - 1) / kBnCols4;
  const int parts = bn_parts(rows, gx);
  const long long rows_per_part = (rows + parts - 1) / parts;
  bn_stats_partial_kernel<<<dim3(gx, parts), kBnThreads, 0, stream>>>(v, rows, C, v_ld, rows_per_part, scratch,
                                                                      num_batches_tracked);
  AVC_CHECK_CUDA(cudaGetLastError());
  bn_stats_final_kernel<<<(C + 31) / 32, kBnThreads, 0, stream>>>(scratch, parts, rows, C, gamma, beta, eps, momentum,
                                                                  cumulative, running_mean, running_var,
                                                                  num_batches_tracked, scale_shift);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch(2);
  return 0;
}

extern "C" int avc_bn_apply(const avc_bn_apply_desc* d, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d && d->v && d->scale_shift && (d->out || d->out2), "avc_bn_apply: null buffer");
  const long long rows = (long long)d->B * d->T;
  AVC_REQUIRE(d->B > 0 && d->T > 0 && rows < (1LL << 31) && d->C > 0 && d->C % 4 == 0 && d->v_ld >= d->C &&
                  d->v_ld % 4 == 0,
              "avc_bn_apply: bad shape B=%d T=%d C=%d", d->B, d->T, d->C);
  AVC_REQUIRE(d->act == AVC_ACT_NONE || d->act == AVC_ACT_RELU || d->act == AVC_ACT_TANH,
              "avc_bn_apply: act %d (NONE / RELU / TANH)", d->act);
  AVC_REQUIRE(!d->residual || (d->res_ld >= d->C && d->res_ld % 4 == 0), "avc_bn_apply: residual ld");
  AVC_REQUIRE(!d->out2 || (d->out2_ld >= d->C && d->out2_ld % 4 == 0), "avc_bn_apply: out2 ld");
  if (d->out) {
    AVC_REQUIRE(d->out_dtype >= 0 && d->out_dtype <= 4 && d->out_ld >= op_ld(d->C, d->out_dtype) && d->out_ld % 4 == 0 &&
                    d->out_row0 >= 0 && d->out_rows_per_utt >= d->out_row0 + d->T,
                "avc_bn_apply: bad out (dtype %d, ld %lld, rows %d, row0 %d)", d->out_dtype, d->out_ld,
                d->out_rows_per_utt, d->out_row0);
  }
  const int gx = (d->C / 4 + kBnCols4 - 1) / kBnCols4;
  long long gy = (rows + kBnRowLanes - 1) / kBnRowLanes;
  const long long cap = (8LL * num_sms() + gx - 1) / gx;   // about eight CTAs per SM, a few rows per thread
  if (gy > cap) gy = cap;
  bn_apply_kernel<<<dim3(gx, (unsigned)gy), kBnThreads, 0, stream>>>(*d);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}
