// HBM-bound glue and the small-H bidirectional LSTM (see include/avc_b200.h).
#include <cuda_bf16.h>

#include <cstdlib>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"
#include "avc_store.cuh"

namespace avc {

// ---------------------------------------------------------------------------------------------
// concat with broadcast: out[b,t,:] = [seq[b, t/div, :C1] || vec[b, :C2]], float4 granularity
// ---------------------------------------------------------------------------------------------
template <int MODE>   // 0 fp32 (optionally TF32-rounded), 1 bf16, 2 split bf16 [hi | lo], 3 fp16
__global__ void __launch_bounds__(256) concat_bcast_kernel(const float* __restrict__ seq, const float* __restrict__ vec,
                                                           void* __restrict__ out, long long rows, int T, int C1,
                                                           int C2, int div, int round) {
  const int c4 = (C1 + C2) >> 2;   // float4 groups per output row
  const long long total = rows * c4;
  const int Tin = T / div;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / c4;
    const int c = static_cast<int>(i - r * c4) << 2;
    const long long b = r / T;
    const int t = static_cast<int>(r - b * T);
    float4 v;
    if (c < C1)   // C2 == 0: pure conversion of seq
      v = __ldg(reinterpret_cast<const float4*>(seq + (b * Tin + t / div) * C1 + c));
    else
      v = __ldg(reinterpret_cast<const float4*>(vec + b * C2 + (c - C1)));
    if (MODE == 2) {
      const int C = C1 + C2;
      __nv_bfloat16* base = static_cast<__nv_bfloat16*>(out) + r * (2LL * C) + c;
      const float lx = v.x - __bfloat162float(__float2bfloat16_rn(v.x));
      const float ly = v.y - __bfloat162float(__float2bfloat16_rn(v.y));
      const float lz = v.z - __bfloat162float(__float2bfloat16_rn(v.z));
      const float lw = v.w - __bfloat162float(__float2bfloat16_rn(v.w));
      *reinterpret_cast<uint2*>(base) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
      *reinterpret_cast<uint2*>(base + C) = make_uint2(pack_bf16(lx, ly), pack_bf16(lz, lw));
    } else if (MODE == 1) {
      uint2 pk = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
      *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(out) + r * (C1 + C2) + c) = pk;
    } else if (MODE == 3) {
      uint2 pk = make_uint2(pack_f16(v.x, v.y), pack_f16(v.z, v.w));
      *reinterpret_cast<uint2*>(static_cast<__half*>(out) + r * (C1 + C2) + c) = pk;
    } else {
      if (round) v = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
      *reinterpret_cast<float4*>(static_cast<float*>(out) + r * (C1 + C2) + c) = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// small-H bidirectional LSTM: one warp per (utterance, direction); W_hh transposed in shared memory
// as Wt[dir][k][unit][gate] so that a lane's four gate weights for input k are one 16-byte load and the
// 32 lanes of a warp read consecutive units (conflict free); h_{t-1} is broadcast from shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int kSmallWarps = 8;   // 4 utterances x 2 directions per CTA

// Padded utterance (Tb < T valid frames): direction `dir`'s half of out rows Tb..T-1 and of codes Tb/freq..T/freq-1 is
// written as 0, by `nthreads` threads of index `tid`.  Zero is all-zero bits in every out_mode.
__device__ __noinline__ void zero_bilstm_tail(void* out, int out_mode, float* codes, int b, int T, int H, int freq, int Tb,
                                              int dir, int tid, int nthreads) {
  if (out) {
    const int es = out_mode == 0 ? 4 : 2;
    const int parts = out_mode == 2 ? 2 : 1;               // split bf16: [hi(2H) | lo(2H)]
    char* base = static_cast<char*>(out);
    for (int i = tid; i < (T - Tb) * parts * H; i += nthreads) {
      const int u = i % H, part = (i / H) % parts, t = Tb + i / (H * parts);
      const long long e = ((long long)b * T + t) * (2LL * parts * H) + part * 2 * H + dir * H + u;
      if (es == 4) reinterpret_cast<float*>(base)[e] = 0.0f; else reinterpret_cast<unsigned short*>(base)[e] = 0;
    }
  }
  if (codes) {
    const int n_codes = T / freq;
    for (int i = tid; i < (n_codes - Tb / freq) * H; i += nthreads)
      codes[((long long)b * n_codes + Tb / freq + i / H) * (2LL * H) + dir * H + i % H] = 0.0f;
  }
}

// REGW (H == 32 only): every lane keeps the 4 x 32 recurrent weights of its hidden unit in registers and h_{t-1} is
// exchanged with warp shuffles, so a step issues 32 SHFL + 128 FMA instead of 64 shared-memory loads (the shared-memory
// variant is bound by those loads: 2.2 K cycles per step against ~0.6 K here).
template <int UPL, bool REGW>   // hidden units per lane: 1 (H <= 32) or 2 (H <= 64)
__global__ void __launch_bounds__(kSmallWarps * 32) bilstm_small_kernel(
    const float* __restrict__ xproj, const float* __restrict__ w_hh, void* __restrict__ out, int out_mode, int round,
    float* __restrict__ codes, int B, int T, int H, int freq, const int* __restrict__ lengths) {
  extern __shared__ float4 smem4[];
  constexpr int HP = UPL * 32;
  float4* Wt = smem4;                                              // [2][H][HP]
  float* hbuf = reinterpret_cast<float*>(smem4 + 2 * H * HP);      // [kSmallWarps][HP]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 2 * H * HP; i += blockDim.x) {
    const int u = i % HP;
    const int k = (i / HP) % H;
    const int d = i / (HP * H);
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
    if (u < H) {
      const float* base = w_hh + (long long)d * 4 * H * H;
      w.x = base[(0 * H + u) * H + k];
      w.y = base[(1 * H + u) * H + k];
      w.z = base[(2 * H + u) * H + k];
      w.w = base[(3 * H + u) * H + k];
    }
    Wt[i] = w;
  }
  float* hb = hbuf + warp * HP;
  for (int e = 0; e < UPL; ++e) hb[lane + 32 * e] = 0.0f;
  __syncthreads();

  const int b = blockIdx.x * (kSmallWarps / 2) + (warp >> 1);
  const int dir = warp & 1;
  if (b >= B) return;          // no CTA barrier past this point: the 4 utterances of a CTA may differ in length
  const float4* W = Wt + dir * H * HP;
  const int n_codes = T / freq;
  const int Tb = lengths ? __ldg(lengths + b) : T;   // valid frames of this utterance
  float c[UPL];
  float zx[UPL][4];
  for (int e = 0; e < UPL; ++e) c[e] = 0.0f;

  auto load_x = [&](int t, float (&dst)[UPL][4]) {
    const float* xp = xproj + ((long long)b * T + t) * (8LL * H) + dir * 4 * H;
#pragma unroll
    for (int e = 0; e < UPL; ++e) {
      const int u = lane + 32 * e;
#pragma unroll
      for (int g = 0; g < 4; ++g) dst[e][g] = (u < H) ? __ldg(xp + g * H + u) : 0.0f;
    }
  };
  load_x(dir ? Tb - 1 : 0, zx);
  float4 wreg[REGW ? 32 : 1];
  float hprev = 0.0f;
  if (REGW) {
#pragma unroll
    for (int k = 0; k < 32; ++k) wreg[k] = W[k * HP + lane];
  }
  for (int s = 0; s < Tb; ++s) {
    const int t = dir ? Tb - 1 - s : s;
    float z[UPL][4];
#pragma unroll
    for (int e = 0; e < UPL; ++e)
#pragma unroll
      for (int g = 0; g < 4; ++g) z[e][g] = zx[e][g];
    if (s + 1 < Tb) load_x(dir ? t - 1 : t + 1, zx);   // prefetch the next frame's projection
    if (REGW) {
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float hk = __shfl_sync(0xffffffffu, hprev, k);
        z[0][0] = fmaf(wreg[k].x, hk, z[0][0]);
        z[0][1] = fmaf(wreg[k].y, hk, z[0][1]);
        z[0][2] = fmaf(wreg[k].z, hk, z[0][2]);
        z[0][3] = fmaf(wreg[k].w, hk, z[0][3]);
      }
    } else {
#pragma unroll 4
      for (int k = 0; k < H; ++k) {
        const float hk = hb[k];
#pragma unroll
        for (int e = 0; e < UPL; ++e) {
          const float4 w = W[k * HP + lane + 32 * e];
          z[e][0] = fmaf(w.x, hk, z[e][0]);
          z[e][1] = fmaf(w.y, hk, z[e][1]);
          z[e][2] = fmaf(w.z, hk, z[e][2]);
          z[e][3] = fmaf(w.w, hk, z[e][3]);
        }
      }
      __syncwarp();
    }
    float h[UPL];
#pragma unroll
    for (int e = 0; e < UPL; ++e) {
      const float ig = sigmoid_fast(z[e][0]);
      const float fg = sigmoid_fast(z[e][1]);
      const float gg = tanh_fast(z[e][2]);
      const float og = sigmoid_fast(z[e][3]);
      c[e] = fg * c[e] + ig * gg;
      h[e] = og * tanh_fast(c[e]);
      if (!REGW) hb[lane + 32 * e] = h[e];
    }
    if (REGW) hprev = h[0]; else __syncwarp();
#pragma unroll
    for (int e = 0; e < UPL; ++e) {
      const int u = lane + 32 * e;
      if (u < H) {
        if (out) {
          const long long o = ((long long)b * T + t) * (2LL * H) + dir * H + u;
          if (out_mode == 2) {   // split bf16: [hi(2H) | lo(2H)]
            const __nv_bfloat16 hi = __float2bfloat16_rn(h[e]);
            __nv_bfloat16* base = static_cast<__nv_bfloat16*>(out) + ((long long)b * T + t) * (4LL * H) + dir * H + u;
            base[0] = hi;
            base[2 * H] = __float2bfloat16_rn(h[e] - __bfloat162float(hi));
          } else if (out_mode == 1)
            static_cast<__nv_bfloat16*>(out)[o] = __float2bfloat16_rn(h[e]);
          else if (out_mode == 3)
            static_cast<__half*>(out)[o] = __float2half_rn(sat_f16(h[e]));
          else
            static_cast<float*>(out)[o] = round ? round_tf32(h[e]) : h[e];
        }
        if (codes) {
          // code_j = [h_fwd[j*freq + freq-1] || h_bwd[j*freq]]  (factory/AutoVC.py:56-66)
          const int r = t % freq;
          if (dir == 0 ? (r == freq - 1) : (r == 0))
            codes[((long long)b * n_codes + t / freq) * (2LL * H) + dir * H + u] = h[e];
        }
      }
    }
  }
  if (Tb < T) zero_bilstm_tail(out, out_mode, codes, b, T, H, freq, Tb, dir, lane, 32);
}

// ---------------------------------------------------------------------------------------------
// H == 32 (AutoVC "A"): FOUR lanes per hidden unit, one CTA of 4 warps per (utterance, direction).
// ncu on the warp-per-(utterance, direction) kernel above: a step is ~365 instructions of ONE warp at an IPC of 0.5 --
// fixed-latency dependencies (32 shuffles + 128 FMAs + the cell) that nothing hides, 1.1 K cycles per step whatever the
// batch is.  Here lane (u, p) keeps the weights of its unit's four gates for the 8 inputs k = 8 p .. 8 p + 7 in registers
// (32 floats), reads those 8 values of h_{t-1} from shared memory (two 16-byte broadcast loads), and the four partial
// sums of a unit meet in two butterfly shuffles; all four lanes then run the cell redundantly (no divergence, c replicated)
// and lane p = 0 publishes h_t.  The serial chain of a step is ~90 instructions instead of ~365.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) bilstm32_kernel(const float* __restrict__ xproj, const float* __restrict__ w_hh,
                                                       void* __restrict__ out, int out_mode, int round,
                                                       float* __restrict__ codes, int T, int freq,
                                                       const int* __restrict__ lengths) {
  constexpr int H = 32;
  __shared__ __align__(16) float hb[2][H];
  const int tid = threadIdx.x;
  const int u = tid >> 2, part = tid & 3;
  const int b = blockIdx.x >> 1, dir = blockIdx.x & 1;
  // w[g][j] = W_hh[dir][g * H + u][8 part + j]
  float w[4][8];
  {
    const float* base = w_hh + (long long)dir * 4 * H * H;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(base + (g * H + u) * H + 8 * part));
      const float4 c4 = __ldg(reinterpret_cast<const float4*>(base + (g * H + u) * H + 8 * part + 4));
      w[g][0] = a.x; w[g][1] = a.y; w[g][2] = a.z; w[g][3] = a.w;
      w[g][4] = c4.x; w[g][5] = c4.y; w[g][6] = c4.z; w[g][7] = c4.w;
    }
  }
  if (tid < 2 * H) (&hb[0][0])[tid] = 0.0f;
  __syncthreads();
  const int n_codes = T / freq;
  const int Tb = lengths ? __ldg(lengths + b) : T;   // valid frames of this utterance (uniform over the CTA)
  // this lane adds the input projection of gate `part` of its unit to its partial sum (the butterfly spreads it)
  const float* xp = xproj + (long long)b * T * (8LL * H) + dir * 4 * H + part * H + u;
  auto frame = [&](int s) { return dir ? Tb - 1 - s : s; };
  constexpr int kPre = 4;                      // projections in flight
  float xq[kPre];
#pragma unroll
  for (int i = 0; i < kPre; ++i) xq[i] = i < Tb ? __ldg(xp + (long long)frame(i) * (8LL * H)) : 0.0f;
  float c = 0.0f;
  for (int s0 = 0; s0 < Tb; s0 += kPre) {
#pragma unroll
    for (int i = 0; i < kPre; ++i) {
      const int s = s0 + i;
      if (s >= Tb) break;
      const int t = frame(s);
      const float xv = xq[i];
      if (s + kPre < Tb) xq[i] = __ldg(xp + (long long)frame(s + kPre) * (8LL * H));
      const float4 h0 = *reinterpret_cast<const float4*>(&hb[s & 1][8 * part]);
      const float4 h1 = *reinterpret_cast<const float4*>(&hb[s & 1][8 * part + 4]);
      const float hk[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
      float z[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float a = g == part ? xv : 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) a = fmaf(w[g][j], hk[j], a);
        z[g] = a;
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        z[g] += __shfl_xor_sync(0xffffffffu, z[g], 1);
        z[g] += __shfl_xor_sync(0xffffffffu, z[g], 2);
      }
      float cn, hn;
      lstm_cell(z[0], z[1], z[2], z[3], c, cn, hn);
      c = cn;
      if (part == 0) {
        hb[(s + 1) & 1][u] = hn;
        if (out) {
          const long long o = ((long long)b * T + t) * (2LL * H) + dir * H + u;
          if (out_mode == 2) {   // split bf16: [hi(2H) | lo(2H)]
            const __nv_bfloat16 hi = __float2bfloat16_rn(hn);
            __nv_bfloat16* ob = static_cast<__nv_bfloat16*>(out) + ((long long)b * T + t) * (4LL * H) + dir * H + u;
            ob[0] = hi;
            ob[2 * H] = __float2bfloat16_rn(hn - __bfloat162float(hi));
          } else if (out_mode == 1)
            static_cast<__nv_bfloat16*>(out)[o] = __float2bfloat16_rn(hn);
          else if (out_mode == 3)
            static_cast<__half*>(out)[o] = __float2half_rn(sat_f16(hn));
          else
            static_cast<float*>(out)[o] = round ? round_tf32(hn) : hn;
        }
        if (codes) {
          // code_j = [h_fwd[j*freq + freq-1] || h_bwd[j*freq]]  (factory/AutoVC.py:56-66)
          const int r = t % freq;
          if (dir == 0 ? (r == freq - 1) : (r == 0))
            codes[((long long)b * n_codes + t / freq) * (2LL * H) + dir * H + u] = hn;
        }
      }
      __syncthreads();      // h_t complete (and every lane done with h_{t-1}) before the next step
    }
  }
  if (Tb < T) zero_bilstm_tail(out, out_mode, codes, b, T, H, freq, Tb, dir, tid, 128);
}

// ---------------------------------------------------------------------------------------------
// LstmDV tail: e = W h + b; out = e / ||e||   one CTA per utterance, one thread per output
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) linear_l2norm_kernel(const float* __restrict__ h, const float* __restrict__ w,
                                                            const float* __restrict__ bias, float* __restrict__ out,
                                                            float* __restrict__ out_raw, int K, int N) {
  extern __shared__ float sh[];   // [K] input row, then 8 partial sums
  float* red = sh + K;
  const int b = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) sh[k] = h[(long long)b * K + k];
  __syncthreads();
  float sq = 0.0f;
  float e_val[4];   // up to N = 1024 outputs with 256 threads
  int cnt = 0;
  for (int n = threadIdx.x; n < N; n += blockDim.x, ++cnt) {
    const float4* wr = reinterpret_cast<const float4*>(w + (long long)n * K);
    float acc = bias[n];
    for (int k = 0; k < K / 4; ++k) {
      const float4 wv = __ldg(wr + k);
      acc = fmaf(wv.x, sh[4 * k], acc);
      acc = fmaf(wv.y, sh[4 * k + 1], acc);
      acc = fmaf(wv.z, sh[4 * k + 2], acc);
      acc = fmaf(wv.w, sh[4 * k + 3], acc);
    }
    e_val[cnt] = acc;
    sq += acc * acc;
  }
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
  __syncthreads();
  float tot = 0.0f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
  const float inv = rsqrtf(tot);
  cnt = 0;
  for (int n = threadIdx.x; n < N; n += blockDim.x, ++cnt) {
    if (out) out[(long long)b * N + n] = e_val[cnt] * inv;
    if (out_raw) out_raw[(long long)b * N + n] = e_val[cnt];
  }
}

// ---------------------------------------------------------------------------------------------
// (B, C, L) fp32 channels-first -> channels-last operand format with reflected halo rows
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void store1(void* out, int mode, int round, long long row, int ld, int c, int C, float v) {
  if (mode == 2) {
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    __nv_bfloat16* p = static_cast<__nv_bfloat16*>(out) + row * ld + c;
    p[0] = hi;
    p[C] = __float2bfloat16_rn(v - __bfloat162float(hi));
  } else if (mode == 4) {
    const __half hi = __float2half_rn(sat_f16(v));
    __half* p = static_cast<__half*>(out) + row * ld + c;
    p[0] = hi;
    p[C] = __float2half_rn(f16_lo(v));
  } else if (mode == 1) {
    static_cast<__nv_bfloat16*>(out)[row * ld + c] = __float2bfloat16_rn(v);
  } else if (mode == 3) {
    static_cast<__half*>(out)[row * ld + c] = __float2half_rn(sat_f16(v));
  } else {
    static_cast<float*>(out)[row * ld + c] = round ? round_tf32(v) : v;
  }
}

__global__ void __launch_bounds__(256) transpose_pad_kernel(const float* __restrict__ in, void* __restrict__ out, int C,
                                                            int L, int pad, int mode, int round) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int l0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {          // coalesced along L
    const int c = c0 + i, l = l0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && l < L) ? __ldg(in + ((long long)b * C + c) * L + l) : 0.0f;
  }
  __syncthreads();
  const int ld = (mode == 2 || mode == 4) ? 2 * C : C;
  const long long base = (long long)b * (L + 2 * pad) + pad;
  for (int i = threadIdx.y; i < 32; i += 8) {          // coalesced along C
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (l < L && c < C) {
      const float v = tile[threadIdx.x][i];
      store1(out, mode, round, base + l, ld, c, C, v);
      if (l >= 1 && l <= pad) store1(out, mode, round, base - l, ld, c, C, v);
      if (l <= L - 2 && l >= L - 1 - pad) store1(out, mode, round, base + 2LL * (L - 1) - l, ld, c, C, v);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// MelGAN output layer: reflect-pad + K-tap conv to one channel + tanh.  One thread per output sample; the
// (256 + K - 1) x C input window of a CTA is staged in shared memory (row stride C+1: conflict free).
// ---------------------------------------------------------------------------------------------
constexpr int kMonoTile = 256;
__global__ void __launch_bounds__(kMonoTile) conv_to_mono_tanh_kernel(const float* __restrict__ x,
                                                                      const float* __restrict__ w, float bias,
                                                                      float* __restrict__ out, int L, int C, int K,
                                                                      const int* __restrict__ lengths) {
  extern __shared__ float sm[];
  const int half = K / 2;
  const int rows = kMonoTile + K - 1;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kMonoTile;
  const int len = lengths ? __ldg(lengths + b) : L;     // a padded batch: reflect at the utterance's end, 0 past it
  if (t0 >= len) {
    if (t0 + (int)threadIdx.x < L) out[(long long)b * L + t0 + threadIdx.x] = 0.f;
    return;
  }
  // rows of C + 4 floats: 16-byte aligned, and consecutive rows start 4 banks apart, so the float4 reads of a quarter
  // warp (8 threads, one row each, same column) cover all 32 banks once -- the kernel is HBM-bound only when it issues
  // 16-byte shared-memory loads (scalar loads made it LDS-bound at 29 % of the HBM peak, ncu r02)
  const int ldx = C + 4;
  float* xs = sm;                       // [rows][C + 4]
  float* ws = sm + rows * ldx;          // [K][C]
  for (int i = threadIdx.x; i < K * C; i += blockDim.x) ws[i] = w[i];
  const int c4 = C / 4;
  for (int i = threadIdx.x; i < rows * c4; i += blockDim.x) {
    const int r = i / c4, c = (i - r * c4) * 4;
    int src = t0 + r - half;
    if (src < 0) src = -src;                         // ReflectionPad1d: edge sample not repeated
    if (src >= len) src = 2 * (len - 1) - src;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (src >= 0 && src < len) v = __ldg(reinterpret_cast<const float4*>(x + ((long long)b * L + src) * C + c));
    *reinterpret_cast<float4*>(xs + r * ldx + c) = v;
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= L) return;
  if (t >= len) {
    out[(long long)b * L + t] = 0.f;
    return;
  }
  float acc0 = bias, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
  for (int k = 0; k < K; ++k) {
    const float4* xr = reinterpret_cast<const float4*>(xs + (threadIdx.x + k) * ldx);
    const float4* wr = reinterpret_cast<const float4*>(ws + k * C);
#pragma unroll 8
    for (int c = 0; c < c4; ++c) {
      const float4 xv = xr[c], wv = wr[c];
      acc0 = fmaf(xv.x, wv.x, acc0);
      acc1 = fmaf(xv.y, wv.y, acc1);
      acc2 = fmaf(xv.z, wv.z, acc2);
      acc3 = fmaf(xv.w, wv.w, acc3);
    }
  }
  const float acc = (acc0 + acc1) + (acc2 + acc3);
  out[(long long)b * L + t] = tanh_fast(acc);
}

}  // namespace avc

extern "C" int avc_concat_bcast(const float* seq, const float* vec, void* out, int B, int T, int C1, int C2, int div,
                                int out_dtype, int out_round_tf32, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(seq && out && (vec || C2 == 0), "avc_concat_bcast: null buffer");
  AVC_REQUIRE(B > 0 && T > 0 && C1 > 0 && C2 >= 0 && C1 % 4 == 0 && C2 % 4 == 0 && div > 0 && T % div == 0,
              "avc_concat_bcast: bad shape B=%d T=%d C1=%d C2=%d div=%d", B, T, C1, C2, div);
  const long long rows = (long long)B * T;
  const long long total = rows * ((C1 + C2) / 4);
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  AVC_REQUIRE(out_dtype >= 0 && out_dtype <= 3, "avc_concat_bcast: out_dtype %d", out_dtype);
  if (out_dtype == 3)
    concat_bcast_kernel<3><<<(int)blocks, 256, 0, stream>>>(seq, vec, out, rows, T, C1, C2, div, 0);
  else if (out_dtype == 2)
    concat_bcast_kernel<2><<<(int)blocks, 256, 0, stream>>>(seq, vec, out, rows, T, C1, C2, div, 0);
  else if (out_dtype == 1)
    concat_bcast_kernel<1><<<(int)blocks, 256, 0, stream>>>(seq, vec, out, rows, T, C1, C2, div, 0);
  else
    concat_bcast_kernel<0><<<(int)blocks, 256, 0, stream>>>(seq, vec, out, rows, T, C1, C2, div, out_round_tf32);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_bilstm_small(const float* xproj, const float* w_hh, void* out, int out_dtype, int out_round_tf32,
                                float* codes, int B, int T, int H, int freq, void* stream_v, const int* lengths) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(xproj && w_hh && (out || codes), "avc_bilstm_small: null buffer");
  AVC_REQUIRE(B > 0 && T > 0 && H > 0 && H <= 64, "avc_bilstm_small: bad shape B=%d T=%d H=%d", B, T, H);
  if (codes) AVC_REQUIRE(freq > 0 && T % freq == 0, "avc_bilstm_small: T=%d is not a multiple of freq=%d", T, freq);
  if (freq <= 0) freq = 1;
  const int upl = H <= 32 ? 1 : 2;
  const int hp = upl * 32;
  const size_t smem = (size_t)2 * H * hp * sizeof(float4) + (size_t)kSmallWarps * hp * sizeof(float);
  const int grid = (B + kSmallWarps / 2 - 1) / (kSmallWarps / 2);
  // four lanes per unit: a 2.9x shorter dependent chain per step, four times the warps.  Measured (T = 1024 / 128, two
  // layers): B = 1 1.15 -> 0.78 ms, B = 32 1.47 -> 0.79 ms, but B = 512 0.21 -> 0.24 ms (issue-bound there): small batches only
  static const bool lanes4 = getenv("AVC_BILSTM_WARP") == nullptr;   // AVC_BILSTM_WARP=1: the warp-per-direction kernel (A/B timing)
  if (H == 32 && lanes4 && B <= 128) {
    bilstm32_kernel<<<2 * B, 128, 0, stream>>>(xproj, w_hh, out, out_dtype, out_round_tf32, codes, T, freq, lengths);
  } else if (H == 32) {   // AutoVC "A" (dim_neck = 32): recurrent weights in registers
    auto kern = bilstm_small_kernel<1, true>;
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kSmallWarps * 32, smem, stream>>>(xproj, w_hh, out, out_dtype, out_round_tf32, codes, B, T, H, freq, lengths);
  } else if (upl == 1) {
    auto kern = bilstm_small_kernel<1, false>;
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kSmallWarps * 32, smem, stream>>>(xproj, w_hh, out, out_dtype, out_round_tf32, codes, B, T, H, freq, lengths);
  } else {
    auto kern = bilstm_small_kernel<2, false>;
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kSmallWarps * 32, smem, stream>>>(xproj, w_hh, out, out_dtype, out_round_tf32, codes, B, T, H, freq, lengths);
  }
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_linear_l2norm(const float* h, const float* w, const float* bias, float* out, int B, int K, int N,
                                 void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(h && w && bias && out, "avc_linear_l2norm: null buffer");
  AVC_REQUIRE(B > 0 && K > 0 && K % 4 == 0 && N > 0 && N <= 1024, "avc_linear_l2norm: bad shape B=%d K=%d N=%d", B, K, N);
  linear_l2norm_kernel<<<B, 256, (K + 8) * sizeof(float), stream>>>(h, w, bias, out, nullptr, K, N);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_linear_rows(const float* h, const float* w, const float* bias, float* out_raw, float* out_normed,
                               int B, int K, int N, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(h && w && bias && (out_raw || out_normed), "avc_linear_rows: null buffer");
  AVC_REQUIRE(B > 0 && K > 0 && K % 4 == 0 && N > 0 && N <= 1024, "avc_linear_rows: bad shape B=%d K=%d N=%d", B, K, N);
  linear_l2norm_kernel<<<B, 256, (K + 8) * sizeof(float), stream>>>(h, w, bias, out_normed, out_raw, K, N);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_transpose_pad(const float* in, void* out, int B, int C, int L, int pad, int out_dtype,
                                 int out_round_tf32, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(in && out, "avc_transpose_pad: null buffer");
  AVC_REQUIRE(B > 0 && C > 0 && C % 4 == 0 && L > pad && pad >= 0 && B < 65536, "avc_transpose_pad: bad shape B=%d C=%d L=%d pad=%d",
              B, C, L, pad);
  AVC_REQUIRE(out_dtype >= 0 && out_dtype <= 4, "avc_transpose_pad: out_dtype %d", out_dtype);
  dim3 grid((L + 31) / 32, (C + 31) / 32, B);
  transpose_pad_kernel<<<grid, dim3(32, 8), 0, stream>>>(in, out, C, L, pad, out_dtype, out_round_tf32);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Reflected halo rows of a channels-last buffer (nn.ReflectionPad1d of the consumer, melgan/modules.py:77,96,121)
// ---------------------------------------------------------------------------------------------
namespace avc {
__global__ void __launch_bounds__(256) reflect_halo_kernel(uint4* __restrict__ buf, long long rows_per_utt, int vec_per_row,
                                                           long long row0, long long L, int reflect, long long total,
                                                           const int* __restrict__ lengths) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = static_cast<int>(i % vec_per_row);
    long long r = i / vec_per_row;
    const int k = static_cast<int>(r % (2 * reflect));       // 0..reflect-1: left halo row -(k+1); rest: right halo
    const long long b = r / (2 * reflect);
    long long dst, src;
    if (k < reflect) {
      dst = row0 - (k + 1);
      src = row0 + (k + 1);
    } else {
      const int j = k - reflect + 1;
      const long long end = lengths ? (long long)__ldg(lengths + b) : L;    // the utterance's own last row
      dst = row0 + end - 1 + j;
      src = row0 + end - 1 - j;
    }
    uint4* base = buf + b * rows_per_utt * vec_per_row;
    base[dst * vec_per_row + v] = base[src * vec_per_row + v];
  }
}
}  // namespace avc

extern "C" int avc_reflect_halo(void* buf, int B, int rows_per_utt, long long row_bytes, int row0, int L, int reflect,
                                void* stream_v, const int* lengths) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(buf != nullptr, "avc_reflect_halo: null buffer");
  AVC_REQUIRE(B > 0 && reflect >= 1 && L > reflect && row0 >= reflect && rows_per_utt >= row0 + L + reflect &&
                  row_bytes > 0 && row_bytes % 16 == 0,
              "avc_reflect_halo: bad geometry B=%d rows=%d row_bytes=%lld row0=%d L=%d reflect=%d", B, rows_per_utt,
              row_bytes, row0, L, reflect);
  const int vec = static_cast<int>(row_bytes / 16);
  const long long total = (long long)B * 2 * reflect * vec;
  const long long blocks = (total + 255) / 256;
  reflect_halo_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, stream>>>(
      static_cast<uint4*>(buf), rows_per_utt, vec, row0, L, reflect, total, lengths);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Padded tails of a variable-length batch: rows row0 + lengths[b] .. row0 + T - 1 of utterance b set to zero
// ---------------------------------------------------------------------------------------------
namespace avc {
__global__ void __launch_bounds__(256) zero_tail_kernel(uint4* __restrict__ buf, long long rows_per_utt, int vec_per_row,
                                                        int row0, int T, const int* __restrict__ lengths) {
  const int b = blockIdx.y;
  const int len = __ldg(lengths + b);
  const long long total = (long long)(T - len) * vec_per_row;
  uint4* base = buf + (b * rows_per_utt + row0 + len) * vec_per_row;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    base[i] = make_uint4(0u, 0u, 0u, 0u);
}
}  // namespace avc

extern "C" int avc_zero_tail(void* buf, int B, int rows_per_utt, long long row_bytes, int row0, int T, const int* lengths,
                             void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(buf != nullptr && lengths != nullptr, "avc_zero_tail: null buffer");
  AVC_REQUIRE(B > 0 && B <= 65535 && T > 0 && row0 >= 0 && rows_per_utt >= row0 + T && row_bytes > 0 && row_bytes % 16 == 0,
              "avc_zero_tail: bad geometry B=%d rows=%d row_bytes=%lld row0=%d T=%d", B, rows_per_utt, row_bytes, row0, T);
  const int vec = static_cast<int>(row_bytes / 16);
  // enough CTAs per utterance for its longest possible tail; an utterance's CTAs past its own tail exit at once
  const long long per_utt = ((long long)T * vec + 255) / 256;
  const dim3 grid((unsigned)(per_utt < 64 ? per_utt : 64), (unsigned)B);
  zero_tail_kernel<<<grid, 256, 0, stream>>>(static_cast<uint4*>(buf), rows_per_utt, vec, row0, T, lengths);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Audio2Mel front end glue (melgan/modules.py:55-66): reflect padding + framing rows, complex magnitude
// ---------------------------------------------------------------------------------------------
namespace avc {

__global__ void __launch_bounds__(256) audio_frames_kernel(const float* __restrict__ audio, void* __restrict__ out,
                                                           long long L, int pad, int hop, int rows, int mode, int round,
                                                           long long total4) {
  const int c4n = hop >> 2;
  const long long padded = L + 2LL * pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;                     // b * rows + r
    const int c = static_cast<int>(i - row * c4n) << 2;
    const long long b = row / rows;
    const long long r = row - b * rows;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long long j = r * hop + c + e;             // index in the padded signal
      long long src = j - pad;
      if (src < 0) src = -src;                         // F.pad(..., "reflect"): no edge repeat
      if (src >= L) src = 2 * (L - 1) - src;
      v[e] = (j < padded && src >= 0 && src < L) ? __ldg(audio + b * L + src) : 0.0f;
    }
    store_op4(out, mode, round, row, op_ld(hop, mode), c, hop, make_float4(v[0], v[1], v[2], v[3]));
  }
}

__global__ void __launch_bounds__(256) complex_mag_kernel(const float* __restrict__ spec, void* __restrict__ mag,
                                                          int bins, int bins_pad, int mode, int round, long long total4) {
  const int c4n = bins_pad >> 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / c4n;
    const int c = static_cast<int>(i - row * c4n) << 2;
    const float* re = spec + row * (2LL * bins);
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = c + e;
      float m = 0.0f;
      if (k < bins) {
        const float a = __ldg(re + k), b = __ldg(re + bins + k);
        m = sqrtf(a * a + b * b);
      }
      v[e] = m;
    }
    store_op4(mag, mode, round, row, op_ld(bins_pad, mode), c, bins_pad, make_float4(v[0], v[1], v[2], v[3]));
  }
}

static int ew_grid(long long total) {
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  return (int)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

}  // namespace avc

extern "C" int avc_audio_frames(const float* audio, void* out, int B, long long L, int pad, int hop, int rows,
                                int out_dtype, int out_round_tf32, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(audio && out, "avc_audio_frames: null buffer");
  AVC_REQUIRE(B > 0 && L > pad && pad >= 0 && hop > 0 && hop % 8 == 0 && rows > 0 && out_dtype >= 0 && out_dtype <= 3,
              "avc_audio_frames: bad shape B=%d L=%lld pad=%d hop=%d rows=%d", B, L, pad, hop, rows);
  const long long total4 = (long long)B * rows * (hop / 4);
  audio_frames_kernel<<<ew_grid(total4), 256, 0, stream>>>(audio, out, L, pad, hop, rows, out_dtype, out_round_tf32,
                                                           total4);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_complex_mag(const float* spec, void* mag, long long rows, int bins, int bins_pad, int out_dtype,
                               int out_round_tf32, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(spec && mag, "avc_complex_mag: null buffer");
  AVC_REQUIRE(rows > 0 && bins > 0 && bins_pad >= bins && bins_pad % 8 == 0 && out_dtype >= 0 && out_dtype <= 3,
              "avc_complex_mag: bad shape rows=%lld bins=%d bins_pad=%d", rows, bins, bins_pad);
  const long long total4 = rows * (bins_pad / 4);
  complex_mag_kernel<<<ew_grid(total4), 256, 0, stream>>>(spec, mag, bins, bins_pad, out_dtype, out_round_tf32, total4);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

extern "C" int avc_conv_to_mono_tanh(const float* x, const float* w, float bias, float* out, int B, int L, int C, int K,
                                     void* stream_v, const int* lengths) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(x && w && out, "avc_conv_to_mono_tanh: null buffer");
  AVC_REQUIRE(B > 0 && B < 65536 && L > K / 2 && C > 0 && C <= 64 && C % 4 == 0 && K % 2 == 1 && K <= 15,
              "avc_conv_to_mono_tanh: bad shape B=%d L=%d C=%d K=%d", B, L, C, K);
  const size_t smem = ((size_t)(kMonoTile + K - 1) * (C + 4) + (size_t)K * C) * sizeof(float);
  AVC_CHECK_CUDA(cudaFuncSetAttribute(conv_to_mono_tanh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((L + kMonoTile - 1) / kMonoTile, B);
  conv_to_mono_tanh_kernel<<<grid, kMonoTile, smem, stream>>>(x, w, bias, out, L, C, K, lengths);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}
