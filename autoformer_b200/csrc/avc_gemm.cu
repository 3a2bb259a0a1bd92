// Implicit-GEMM convolution / dense GEMM on tcgen05 (see include/avc_b200.h: avc_conv_gemm).
//
// Tile = 128 GEMM rows x BN output columns.  The 128 rows are `bb` utterances x `tb` consecutive frames
// (tb * bb = 128, the power-of-two split that wastes the fewest rows), so one 3-D TMA box
// {128 bytes of channels, tb frames, bb utterances} fetches the A tile of one (source, tap, channel chunk)
// k-block, shifted in time by the tap offset; frames outside the utterance are zero-filled by TMA, which IS
// the convolution's zero padding -- tiles never bleed across utterances.
#include <cuda_bf16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

constexpr int kMaxSrc = AVC_MAX_SOURCES;

struct alignas(64) GemmParams {
  CUtensorMap tmap_a[kMaxSrc];
  CUtensorMap tmap_b;
  // k-block schedule: source s owns k-blocks [kb_end[s-1], kb_end[s]), tap-major, `chunks` channel chunks per tap
  int kb_end[kMaxSrc];
  int chunks[kMaxSrc];
  int tap_t0[kMaxSrc];
  int tap_dt[kMaxSrc];
  int num_kb;
  int kc_elems;          // channels per k-block (32 tf32 / 64 bf16)
  // tiling
  int B, T, N;
  int tb_log2, bb;       // tile = bb utterances x (1 << tb_log2) frames
  int tiles_t, n_tiles;
  int num_units;         // (pairs of) m-tiles x n-tiles; CTAs (pairs) loop over them with stride gridDim.x / CTAS
  // epilogue
  const float* bias;
  int act;
  int phases, cs;        // output time = phases * t + phase0 + n / cs; this launch produces N / cs of the `phases` phases
  int phase0;
  void* out;
  long long out_ld;
  int out_rows_per_utt, out_row0, out_mode, out_round, out_reflect;   // out_mode: 0 fp32, 1 bf16, 2 split bf16, 3 fp16, 4 split fp16
  int raw_mode;           // format of out_raw (same codes)
  uint32_t fmt_xor;       // kIdescF16Xor when the 16-bit operands are fp16
  void* out_raw;
  long long out_raw_ld;
  float* out2;
  long long out2_ld;
  const float* residual;
  long long res_ld;
  int res_after;
  long long* debug_clk;  // optional: 4 clock64 stamps per CTA (entry, setup done, accumulator ready, epilogue done)
};

template <int ACT>
__device__ __forceinline__ float apply_act(float v) {
  if (ACT == AVC_ACT_RELU) return fmaxf(v, 0.0f);
  if (ACT == AVC_ACT_TANH) return tanh_fast(v);
  if (ACT == AVC_ACT_LRELU) return fmaxf(v, 0.2f * v);      // slope < 1
  if (ACT == AVC_ACT_GELU) {
    // exact-erf GELU, 0.5 v (1 + erf(v / sqrt 2)), with erfc(|x|) = t (a1 + t (a2 + ... a5 t)) exp(-x^2), t = 1 / (1 + p |x|)
    // (Abramowitz & Stegun 7.1.26, |error| <= 1.5e-7 -- fp32 rounding level; two MUFU ops and no branch, where erff()
    // costs the low-K mixer GEMMs more than their MMAs).  1 + erf(x) is formed without cancellation on the negative side.
    const float x = fabsf(v) * 0.70710678118654752f;
    const float t = __fdividef(1.0f, fmaf(0.3275911f, x, 1.0f));
    float q = fmaf(t, 1.061405429f, -1.453152027f);
    q = fmaf(t, q, 1.421413741f);
    q = fmaf(t, q, -0.284496736f);
    q = fmaf(t, q, 0.254829592f);
    q = q * t * __expf(-x * x);                       // erfc(|x|)
    return 0.5f * v * (v < 0.0f ? q : 2.0f - q);
  }
  if (ACT == AVC_ACT_LOG10_CLAMP) return log10f(fmaxf(v, 1e-5f));
  return v;
}

// Store four consecutive channels [c, c+4) of one output row in the operand format `mode`.
__device__ __forceinline__ void store4(void* base, int mode, int round, long long row, long long ld, int c, int cs,
                                       const float (&v)[4]) {
  if (mode == 2) {
    float lo[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) lo[i] = v[i] - __bfloat162float(__float2bfloat16_rn(v[i]));
    __nv_bfloat16* ptr = static_cast<__nv_bfloat16*>(base) + row * ld + c;
    *reinterpret_cast<uint2*>(ptr) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
    *reinterpret_cast<uint2*>(ptr + cs) = make_uint2(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]));
  } else if (mode == 4) {
    __half* ptr = static_cast<__half*>(base) + row * ld + c;
    uint2 hi, lo;
    split_f16_pair(v[0], v[1], hi.x, lo.x);
    split_f16_pair(v[2], v[3], hi.y, lo.y);
    *reinterpret_cast<uint2*>(ptr) = hi;
    *reinterpret_cast<uint2*>(ptr + cs) = lo;
  } else if (mode == 1) {
    uint2 pk = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
    *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(base) + row * ld + c) = pk;
  } else if (mode == 3) {
    uint2 pk = make_uint2(pack_f16(v[0], v[1]), pack_f16(v[2], v[3]));
    *reinterpret_cast<uint2*>(static_cast<__half*>(base) + row * ld + c) = pk;
  } else {
    float4 o = round ? make_float4(round_tf32(v[0]), round_tf32(v[1]), round_tf32(v[2]), round_tf32(v[3]))
                     : make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(static_cast<float*>(base) + row * ld + c) = o;
  }
}

// Predicated store of four consecutive channels in a 16-bit operand format (1 bf16, 2 split bf16, 3 fp16, 4 split fp16).
__device__ __forceinline__ void store16(__nv_bfloat16* ptr, int mode, int cs, const float (&o)[4], bool ok) {
  if (mode >= 3) {
    uint2 hi, lo;
    if (mode == 4) {
      split_f16_pair(o[0], o[1], hi.x, lo.x);
      split_f16_pair(o[2], o[3], hi.y, lo.y);
      if (ok) *reinterpret_cast<uint2*>(ptr + cs) = lo;
    } else {
      hi = make_uint2(pack_f16(o[0], o[1]), pack_f16(o[2], o[3]));
    }
    if (ok) *reinterpret_cast<uint2*>(ptr) = hi;
  } else {
    if (ok) *reinterpret_cast<uint2*>(ptr) = make_uint2(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]));
    if (mode == 2) {
      float lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) lo[e] = o[e] - __bfloat162float(__float2bfloat16_rn(o[e]));
      if (ok) *reinterpret_cast<uint2*>(ptr + cs) = make_uint2(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]));
    }
  }
}

// Epilogue of one 128 x BN accumulator tile, run by the kEpiWarps epilogue warps of a CTA.
// tcgen05.ld hands thread i the 32 columns of accumulator ROW i; storing that directly would write 8..16-byte
// fragments of 32 different rows per instruction.  Each 32x32 chunk is therefore transposed through a padded
// shared-memory tile: afterwards 8 consecutive lanes own 32 consecutive channels of ONE row, so every global
// load/store of the epilogue (bias, residual, outputs) is a full 64..128-byte row segment.
// Epilogue warp e (0..7) may touch TMEM lanes [32*(e%4), +32) (hardware rule: warp_id % 4); the two warps of a lane
// quarter take alternate 32-column chunks.
template <int BN, int ACT>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, const PipeSmem& s, uint32_t tmem_base, int ew, int lane,
                                              int b0, int t0, int n0, uint64_t* tmem_empty_bar) {
  const int q = (ew + 2) & 3;            // == warp_id % 4
  const int half = ew >> 2;              // which of the two warps of this quarter
  float* stg = s.staging + ew * (32 * kStagingLd);
  const int cl = (lane & 7) * 4;         // this lane's 4 columns inside a 32-column chunk
  const int rsub = lane >> 3;            // this lane's row inside a group of 4 rows
  const int tb = 1 << p.tb_log2;
  const int t_out = p.T * p.phases;      // output frames per utterance
  const bool has_res = p.residual != nullptr, res_after = p.res_after != 0;
  const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  // 32-column chunks of this tile that hold real output channels.  With a single one (N <= 32: the late MelGAN
  // stages) the two warps of a lane quarter split its ROWS instead of idling one of them.
  const int chunks = min(BN / 32, (p.N - n0 + 31) / 32);
  const bool split_rows = chunks == 1;
  const int c_first = split_rows ? 0 : half;
  const int g_first = split_rows ? half * 4 : 0, g_last = split_rows ? half * 4 + 4 : 8;
  // bias of the first chunk is requested before anything else so its L2 latency overlaps the TMEM load; the bias of
  // chunk c + 2 is requested while chunk c is being stored
  auto load_bias = [&](int c32) {
    const int n = n0 + c32 * 32 + cl;
    return n < p.N ? __ldg(reinterpret_cast<const float4*>(p.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  float4 bv_next = c_first < chunks ? load_bias(c_first) : make_float4(0.f, 0.f, 0.f, 0.f);
  // output shapes served by the branch-free row loops (see below); tiles with one real chunk keep the general loop
  // (poly-phase outputs qualify when a 32-column chunk lies inside one phase; reflected halo rows never do -- callers
  // that want the fast path write them with avc_reflect_halo afterwards)
  int simple = 0;
  if (!split_rows && p.out_reflect == 0 && ((p.phases == 1 && p.phase0 == 0) || (p.cs & 31) == 0)) {
    if (p.out && !p.out2 && !has_res && p.out_mode != 0 && (!p.out_raw || p.raw_mode != 0)) simple = 1;
    if (!p.out && p.out2 && !(has_res && res_after) && p.phases == 1 && !p.out_raw) simple = 2;
  }
  // The row loop is deliberately NOT fully unrolled: with 8 copies of the (mode x output x halo) store code the
  // epilogue was ~4000 instructions, and layers with few k-blocks per tile (MelGAN stages 2-3, 1x1 convolutions) spent
  // 7 K cycles per 32-column chunk fetching instructions (ncu: 20 % stall_no_inst; time per tile independent of K).
#pragma unroll 1
  for (int c32 = c_first; c32 < chunks; c32 += kEpiWarps / 4) {
    uint32_t v[32];
    tmem_ld_32x32(lane_addr + c32 * 32, v);
    tmem_ld_wait();
    if (c32 + kEpiWarps / 4 >= chunks) {    // that was this warp's last read of the accumulator buffer: hand it back
      tc_fence_before();
      if (lane == 0) mbar_arrive_leader(tmem_empty_bar);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      *reinterpret_cast<float4*>(stg + lane * kStagingLd + 4 * j) =
          make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                      __uint_as_float(v[4 * j + 3]));
    __syncwarp();
    const int n = n0 + c32 * 32 + cl;
    const float4 bv = bv_next;
    if (c32 + kEpiWarps / 4 < chunks) bv_next = load_bias(c32 + kEpiWarps / 4);
    if (n < p.N && simple != 0) {
      // The two common output shapes without any per-row branching (the general loop below crosses ~10 branches per
      // 4-element store; with two epilogue warps per scheduler nothing hides their latency, and layers with few
      // k-blocks per tile were bound by it: 13.5 K cycles per 128 x 256 tile against 9 K cycles of MMAs).
      //   simple 1: act(v) to `out` (and optionally v itself to `out_raw`) in 16-bit operand formats, one or two terms
      //   simple 2: act(v [+ residual]) to `out2` (fp32), nothing else
      const int pidx = p.phases == 1 ? 0 : n / p.cs;       // constant over the chunk (cs % 32 == 0)
      const int c = n - pidx * p.cs;
      const int phase = p.phase0 + pidx;
      // NOT unrolled either: eight copies of the body (x six activations) made the kernel 21.6 K SASS instructions and the
      // epilogue warps waited for instruction fetch again (ncu: stall_no_instruction on top) -- measured on the mixers'
      // 344 -> 1376 GEMM at B = 512 (scripts/mixer_unit_timing.py): exact-erf GELU 4.70 ms unrolled x8, 3.64 ms x2,
      // 3.12 ms x1; no activation 2.48 / 2.28 / 2.21 ms; 11.9 K instructions now
      if (p.tb_log2 >= 5) {
        // Tiles of >= 32 frames per utterance (every long-sequence layer): the 32 rows of this lane quarter belong to ONE
        // utterance, so the row part of the address is computed once per chunk and advanced by 4 rows per iteration.
        // The source-level profile of the loop below (profiles/r02_gemm_epilogue_source.txt) shows ~60 instructions per
        // iteration, most of them the (utterance, frame) -> 64-bit offset arithmetic and the branches around the output
        // formats, each waiting on the one before (stall_wait / branch_resolving with two warps per scheduler): 300
        // cycles per iteration, 10 K per 128 x 256 tile whatever the mainloop does.
        const int m0 = q * 32 + rsub;
        const int b = b0 + (m0 >> p.tb_log2);
        const int t = t0 + (m0 & (tb - 1));
        const bool b_ok = b < p.B;
        if (simple == 1) {
          const long long time0 = (long long)t * p.phases + phase;
          __nv_bfloat16* po = static_cast<__nv_bfloat16*>(p.out) + ((long long)b * p.out_rows_per_utt + p.out_row0 + time0) * p.out_ld + c;
          const long long po_step = 4LL * p.phases * p.out_ld;
          if (!p.out_raw && p.out_mode == 3) {
            // one fp16 value per element, nothing else ("fp16x2" activations): the commonest shape gets its own loop
#pragma unroll 2
            for (int i = 0; i < 8; ++i) {
              const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
              const float o0 = apply_act<ACT>(a.x + bv.x), o1 = apply_act<ACT>(a.y + bv.y);
              const float o2 = apply_act<ACT>(a.z + bv.z), o3 = apply_act<ACT>(a.w + bv.w);
              if (b_ok && t + 4 * i < p.T) *reinterpret_cast<uint2*>(po) = make_uint2(pack_f16(o0, o1), pack_f16(o2, o3));
              po += po_step;
            }
          } else if (!p.out_raw && p.out_mode == 4) {
            // two fp16 terms per element, nothing else (MelGAN's "fp16s" residual stream and ConvTranspose outputs)
            __half* ph = reinterpret_cast<__half*>(po);
#pragma unroll 2
            for (int i = 0; i < 8; ++i) {
              const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
              const float o0 = apply_act<ACT>(a.x + bv.x), o1 = apply_act<ACT>(a.y + bv.y);
              const float o2 = apply_act<ACT>(a.z + bv.z), o3 = apply_act<ACT>(a.w + bv.w);
              uint2 hi, lo;
              split_f16_pair(o0, o1, hi.x, lo.x);
              split_f16_pair(o2, o3, hi.y, lo.y);
              if (b_ok && t + 4 * i < p.T) {
                *reinterpret_cast<uint2*>(ph) = hi;
                *reinterpret_cast<uint2*>(ph + p.cs) = lo;
              }
              ph += po_step;
            }
          } else {
            __nv_bfloat16* pr = static_cast<__nv_bfloat16*>(p.out_raw) + ((long long)b * t_out + time0) * p.out_raw_ld + c;
            const long long pr_step = 4LL * p.phases * p.out_raw_ld;
#pragma unroll 1
            for (int i = 0; i < 8; ++i) {
              const bool ok = b_ok && t + 4 * i < p.T;
              const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
              float o[4] = {a.x + bv.x, a.y + bv.y, a.z + bv.z, a.w + bv.w};
              if (p.out_raw) store16(pr, p.raw_mode, p.cs, o, ok);
#pragma unroll
              for (int e = 0; e < 4; ++e) o[e] = apply_act<ACT>(o[e]);
              store16(po, p.out_mode, p.cs, o, ok);
              po += po_step;
              pr += pr_step;
            }
          }
        } else {
          const long long lr0 = (long long)b * p.T + t;
          float* po = p.out2 + lr0 * p.out2_ld + n;
          const float* pres = p.residual + lr0 * p.res_ld + n;
#pragma unroll 2
          for (int i = 0; i < 8; ++i) {
            const bool ok = b_ok && t + 4 * i < p.T;
            const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
            float o[4] = {a.x + bv.x, a.y + bv.y, a.z + bv.z, a.w + bv.w};
            if (has_res) {
              float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
              if (ok) rv = __ldg(reinterpret_cast<const float4*>(pres));
              o[0] += rv.x; o[1] += rv.y; o[2] += rv.z; o[3] += rv.w;
              pres += 4LL * p.res_ld;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) o[e] = apply_act<ACT>(o[e]);
            if (ok) *reinterpret_cast<float4*>(po) = make_float4(o[0], o[1], o[2], o[3]);
            po += 4LL * p.out2_ld;
          }
        }
      } else
#pragma unroll 1
      for (int i = 0; i < 8; ++i) {          // (simple excludes split_rows: all eight row groups are this warp's)
        {
          const int m = q * 32 + 4 * i + rsub;
          const int b = b0 + (m >> p.tb_log2);
          const int t = t0 + (m & (tb - 1));
          const bool ok = b < p.B && t < p.T;
          const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
          float o[4] = {a.x + bv.x, a.y + bv.y, a.z + bv.z, a.w + bv.w};
          if (simple == 1) {
            const int time = t * p.phases + phase;
            if (p.out_raw) {
              __nv_bfloat16* rp = static_cast<__nv_bfloat16*>(p.out_raw) + ((long long)b * t_out + time) * p.out_raw_ld + c;
              store16(rp, p.raw_mode, p.cs, o, ok);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) o[e] = apply_act<ACT>(o[e]);
            const long long off = ((long long)b * p.out_rows_per_utt + p.out_row0 + time) * p.out_ld + c;
            store16(static_cast<__nv_bfloat16*>(p.out) + off, p.out_mode, p.cs, o, ok);   // 2-byte elements in all four formats
          } else {
            const long long lr = (long long)b * p.T + t;
            if (has_res) {
              float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
              if (ok) rv = __ldg(reinterpret_cast<const float4*>(p.residual + lr * p.res_ld + n));
              o[0] += rv.x; o[1] += rv.y; o[2] += rv.z; o[3] += rv.w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) o[e] = apply_act<ACT>(o[e]);
            if (ok) *reinterpret_cast<float4*>(p.out2 + lr * p.out2_ld + n) = make_float4(o[0], o[1], o[2], o[3]);
          }
        }
      }
    } else if (n < p.N) {
      const int pidx = p.phases == 1 ? 0 : n / p.cs;
      const int c = n - pidx * p.cs;
      const int phase = p.phase0 + pidx;
#pragma unroll 2
      for (int i = g_first; i < g_last; ++i) {
        const int m = q * 32 + 4 * i + rsub;
        const int b = b0 + (m >> p.tb_log2);
        const int t = t0 + (m & (tb - 1));
        if (b < p.B && t < p.T) {
          const int time = t * p.phases + phase;
          const long long lr = (long long)b * t_out + time;
          const float4 a = *reinterpret_cast<const float4*>(stg + (4 * i + rsub) * kStagingLd + cl);
          float o[4] = {a.x + bv.x, a.y + bv.y, a.z + bv.z, a.w + bv.w};
          float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (has_res) {
            rv = __ldg(reinterpret_cast<const float4*>(p.residual + lr * p.res_ld + c));
            if (!res_after) { o[0] += rv.x; o[1] += rv.y; o[2] += rv.z; o[3] += rv.w; }
          }
          if (p.out_raw) store4(p.out_raw, p.raw_mode, p.out_round, lr, p.out_raw_ld, c, p.cs, o);
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = apply_act<ACT>(o[e]);
          if (has_res && res_after) { o[0] += rv.x; o[1] += rv.y; o[2] += rv.z; o[3] += rv.w; }
          if (p.out) {
            const long long orw = (long long)b * p.out_rows_per_utt + p.out_row0 + time;
            store4(p.out, p.out_mode, p.out_round, orw, p.out_ld, c, p.cs, o);
            if (p.out_reflect > 0) {   // reflected halo rows (ReflectionPad1d of the consumer); rare: one shared copy
              long long mirror = -1;
              if (time >= 1 && time <= p.out_reflect) mirror = orw - 2LL * time;
              if (mirror >= 0) store4(p.out, p.out_mode, p.out_round, mirror, p.out_ld, c, p.cs, o);
              mirror = -1;
              if (time <= t_out - 2 && time >= t_out - 1 - p.out_reflect) mirror = orw + 2LL * (t_out - 1 - time);
              if (mirror >= 0) store4(p.out, p.out_mode, p.out_round, mirror, p.out_ld, c, p.cs, o);
            }
          }
          if (p.out2) *reinterpret_cast<float4*>(p.out2 + lr * p.out2_ld + c) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    __syncwarp();   // the staging tile is overwritten by the next chunk
  }
  if (c_first >= chunks) {   // a warp without a chunk (cannot happen while every n-tile holds a real column) still hands back
    tc_fence_before();
    if (lane == 0) mbar_arrive_leader(tmem_empty_bar);
  }
}

template <int BN, bool BF16, int CTAS>
__global__ void __launch_bounds__(kNumThreads, 1) conv_gemm_kernel(const __grid_constant__ GemmParams p) {
  // Persistent: each CTA (pair) loops over tile units; the accumulator is double-buffered in tensor memory so the
  // epilogue of unit i runs while the MMAs of unit i+1 are being issued.
  using C = PipeCfg<BN, CTAS, 1, true, 0, 2>;
  extern __shared__ uint8_t smem_raw[];
  const PipeSmem s = carve_smem<C>(smem_raw);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long clk_entry = p.debug_clk ? clock64() : 0;
  // CTA pair: rank 0 (leader) issues the MMAs of the 256-row tile; each CTA owns one 128-row m-tile of it
  const int cta_rank = CTAS == 2 ? (int)cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit0 = blockIdx.x / CTAS;
  const int unit_stride = gridDim.x / CTAS;
  const int tb = 1 << p.tb_log2;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmap_b);
#pragma unroll
    for (int i = 0; i < kMaxSrc; ++i)
      if (i == 0 || p.kb_end[i] > p.kb_end[i - 1]) prefetch_tmap(&p.tmap_a[i]);
  }
  const uint32_t tmem_base = pipe_setup<C>(s);

  // unit -> tile coordinates: n fastest so units processed at the same time share A tiles in L2
  auto coords = [&](int unit, int& b0, int& t0, int& n0) {
    const int n_tile = unit % p.n_tiles;
    const int m_tile = (unit / p.n_tiles) * CTAS + cta_rank;
    t0 = (m_tile % p.tiles_t) * tb;
    b0 = (m_tile / p.tiles_t) * p.bb;
    n0 = n_tile * BN;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer (both CTAs of a pair: own A rows, own half of the B rows)
      RingState rs;
      int itp = 0;
      for (int unit = unit0; unit < p.num_units; unit += unit_stride, ++itp) {
        int b0, t0, n0;
        coords(unit, b0, t0, n0);
        int src = 0, base = 0;
        // per-unit stamps of CTA 0 (profiling aid): 8 slots per unit after the 4-per-CTA block
        long long* ud = (p.debug_clk && blockIdx.x == 0 && itp < 256) ? p.debug_clk + 4LL * gridDim.x + 8 * itp : nullptr;
        if (ud) ud[0] = clock64();                                         // producer starts the unit
        // (Tried and measured slower, r02: L2-prefetching the next unit's activation rows from here with
        // cp.async.bulk.prefetch.tensor -- the up-sampling GEMMs of the long MelGAN stages went from 0.82 to 0.96 ms.
        // Their producer already spends ~700 cycles per k-block ISSUING the two TMA operations of a stage, against 128
        // cycles of MMAs (scripts/up_unit_timing.py): more TMA operations make it worse, not fewer misses better.)
        for (int kb = 0; kb < p.num_kb; ++kb) {
          while (kb >= p.kb_end[src]) {
            base = p.kb_end[src];
            ++src;
          }
          const int local = kb - base;
          const int tap = local / p.chunks[src];
          const int chunk = local - tap * p.chunks[src];
          mbar_wait(&s.empty[rs.stage], rs.phase ^ 1u);
          uint8_t* a_dst = s.base + rs.stage * C::kStageBytes;
          if (CTAS == 2) {
            // all bytes of the pair are credited to the leader's full barrier
            if (leader) mbar_arrive_expect_tx(&s.full[rs.stage], 2 * C::kStageBytes);
            tma_load_3d_2sm(a_dst, &p.tmap_a[src], &s.full[rs.stage], chunk * p.kc_elems,
                            t0 + p.tap_t0[src] + tap * p.tap_dt[src], b0);
            tma_load_2d_2sm(a_dst + kATileBytes, &p.tmap_b, &s.full[rs.stage], kb * p.kc_elems,
                            n0 + cta_rank * (BN / 2));
          } else {
            mbar_arrive_expect_tx(&s.full[rs.stage], C::kStageBytes);
            tma_load_3d(a_dst, &p.tmap_a[src], &s.full[rs.stage], chunk * p.kc_elems,
                        t0 + p.tap_t0[src] + tap * p.tap_dt[src], b0);
            tma_load_2d(a_dst + kATileBytes, &p.tmap_b, &s.full[rs.stage], kb * p.kc_elems, n0);
          }
          rs.advance<C::kStages>();
        }
        if (ud) ud[1] = clock64();                                         // all loads of the unit issued
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      // ---------------- MMA issuer (leader CTA only)
      RingState rs;
      int it = 0;
      for (int unit = unit0; unit < p.num_units; unit += unit_stride, ++it) {
        const int buf = it & 1;
        long long* ud = (p.debug_clk && blockIdx.x == 0 && it < 256) ? p.debug_clk + 4LL * gridDim.x + 8 * it : nullptr;
        if (ud) ud[2] = clock64();                                         // MMA thread reaches the unit
        mbar_wait(&s.tmem_empty[buf], ((it >> 1) & 1) ^ 1u);   // epilogue(s) have drained this accumulator buffer
        tc_fence_after();
        if (ud) ud[3] = clock64();                                         // accumulator buffer free
        const uint32_t acc = tmem_base + buf * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&s.full[rs.stage], rs.phase);
          if (ud && kb == 0) ud[4] = clock64();                            // first k-block landed
          tc_fence_after();
          const uint32_t a_addr = smem_u32(s.base + rs.stage * C::kStageBytes);
          issue_pair<BN, BF16, CTAS>(a_addr, a_addr + kATileBytes, acc, kb == 0, p.fmt_xor);
          // frees the smem slot (in both CTAs of a pair) once these MMAs have read it
          if (CTAS == 2) umma_commit_2sm(&s.empty[rs.stage], 0x3); else umma_commit(&s.empty[rs.stage]);
          rs.advance<C::kStages>();
        }
        if (CTAS == 2) umma_commit_2sm(&s.tmem_full[buf], 0x3); else umma_commit(&s.tmem_full[buf]);
        if (ud) ud[5] = clock64();                                         // all MMAs of the unit issued
      }
    }
  } else {
    // ---------------- epilogue warps
    int it = 0;
    long long clk_first = 0;
    for (int unit = unit0; unit < p.num_units; unit += unit_stride, ++it) {
      int b0, t0, n0;
      coords(unit, b0, t0, n0);
      const int buf = it & 1;
      mbar_wait(&s.tmem_full[buf], (it >> 1) & 1);
      tc_fence_after();
      if (p.debug_clk && it == 0) clk_first = clock64();
      long long* ud = (p.debug_clk && blockIdx.x == 0 && it < 256 && threadIdx.x == 64) ? p.debug_clk + 4LL * gridDim.x + 8 * it : nullptr;
      if (ud) ud[6] = clock64();                                           // accumulator ready (epilogue warp 0)
      const uint32_t acc = tmem_base + buf * BN;
      uint64_t* eb = &s.tmem_empty[buf];
      switch (p.act) {   // the activation is resolved once per tile, not once per element
        case AVC_ACT_RELU: epilogue_tile<BN, AVC_ACT_RELU>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
        case AVC_ACT_TANH: epilogue_tile<BN, AVC_ACT_TANH>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
        case AVC_ACT_LRELU: epilogue_tile<BN, AVC_ACT_LRELU>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
        case AVC_ACT_GELU: epilogue_tile<BN, AVC_ACT_GELU>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
        case AVC_ACT_LOG10_CLAMP: epilogue_tile<BN, AVC_ACT_LOG10_CLAMP>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
        default: epilogue_tile<BN, AVC_ACT_NONE>(p, s, acc, warp - 2, lane, b0, t0, n0, eb); break;
      }
      if (ud) ud[7] = clock64();                                           // epilogue of the unit done (warp 0)
    }
    if (p.debug_clk && threadIdx.x == 64) {
      long long* d = p.debug_clk + 4LL * blockIdx.x;
      d[0] = clk_entry; d[1] = clk_first; d[2] = clock64(); d[3] = it;
    }
  }
  pipe_teardown<C>(tmem_base);
}

template <int BN, bool BF16, int CTAS>
static int launch_impl(const GemmParams& p, long long m_tiles, cudaStream_t stream) {
  auto kern = conv_gemm_kernel<BN, BF16, CTAS>;
  using C = PipeCfg<BN, CTAS, 1, true, 0, 2>;
  static PerDeviceOnce configured;   // per instantiation
  if (configured.first_use()) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes));
  }
  const long long pairs_m = (m_tiles + CTAS - 1) / CTAS;          // a phantom second m-tile is masked in the epilogue
  const long long units = pairs_m * p.n_tiles;
  AVC_REQUIRE(units > 0 && units < (1LL << 30), "avc_conv_gemm: %lld tile units", units);
  GemmParams pp = p;
  pp.num_units = (int)units;
  // persistent: one CTA (pair) per SM (pair), each looping over the units with a fixed stride
  const long long resident = num_sms() / CTAS;
  const long long grid = (units < resident ? units : resident) * CTAS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CTAS > 1 ? 1 : 0;
  AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, pp));
  count_launch();
  return 0;
}

template <int BN, bool BF16>
static int launch(const GemmParams& p, long long m_tiles, int ctas, cudaStream_t stream) {
  return ctas == 2 ? launch_impl<BN, BF16, 2>(p, m_tiles, stream) : launch_impl<BN, BF16, 1>(p, m_tiles, stream);
}

}  // namespace avc

extern "C" int avc_conv_gemm(const avc_gemm_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_conv_gemm: null descriptor");
  AVC_REQUIRE(d->dtype == AVC_DTYPE_TF32 || d->dtype == AVC_DTYPE_BF16 || d->dtype == AVC_DTYPE_F16,
              "avc_conv_gemm: bad dtype %d", d->dtype);
  AVC_REQUIRE(d->B > 0 && d->T > 0 && d->N > 0 && d->N % 4 == 0, "avc_conv_gemm: bad shape B=%d T=%d N=%d", d->B,
              d->T, d->N);
  AVC_REQUIRE(d->a_taps[0] > 0 && d->a_ptr[0] && d->w_ptr && d->bias, "avc_conv_gemm: missing operand");
  AVC_REQUIRE(d->out || d->out2 || d->out_raw, "avc_conv_gemm: no output");
  const int es = d->dtype == AVC_DTYPE_TF32 ? 4 : 2;
  const int kc = kRowBytes / es;

  int bn = d->block_n;
  if (bn == 0) bn = d->n_pad % 256 == 0 ? 256 : (d->n_pad % 128 == 0 ? 128 : 64);
  AVC_REQUIRE(bn == 64 || bn == 128 || bn == 256, "avc_conv_gemm: block_n %d", bn);
  AVC_REQUIRE(d->n_pad % bn == 0 && d->n_pad >= d->N, "avc_conv_gemm: n_pad %d not a multiple of block_n %d", d->n_pad,
              bn);

  GemmParams p;
  memset(&p, 0, sizeof(p));
  // tile = bb utterances x tb frames: pick the power-of-two split of 128 rows that wastes the fewest rows
  int tb_log2 = 7;
  long long best = -1;
  for (int l = 7; l >= 0; --l) {
    const long long tbc = 1LL << l, bbc = kBlockM >> l;
    const long long rows = ((d->T + tbc - 1) / tbc) * ((d->B + bbc - 1) / bbc);
    if (best < 0 || rows < best) {
      best = rows;
      tb_log2 = l;
    }
  }
  const int tb = 1 << tb_log2;
  p.tb_log2 = tb_log2;
  p.bb = kBlockM / tb;
  p.tiles_t = (d->T + tb - 1) / tb;
  const int tiles_b = (d->B + p.bb - 1) / p.bb;
  p.n_tiles = d->n_pad / bn;
  p.B = d->B;
  p.T = d->T;
  p.N = d->N;
  p.kc_elems = kc;

  int kb_total = 0;
  bool ended = false;
  for (int s = 0; s < kMaxSrc; ++s) {
    if (d->a_taps[s] <= 0) {
      ended = true;
      p.kb_end[s] = kb_total;
      p.chunks[s] = 1;
      continue;
    }
    AVC_REQUIRE(!ended, "avc_conv_gemm: sources must be used in order (source %d after an unused one)", s);
    AVC_REQUIRE(d->a_ptr[s] != nullptr, "avc_conv_gemm: source %d null", s);
    p.chunks[s] = (d->a_channels[s] + kc - 1) / kc;
    p.tap_t0[s] = d->a_tap_t0[s];
    p.tap_dt[s] = d->a_tap_dt[s];
    kb_total += d->a_taps[s] * p.chunks[s];
    p.kb_end[s] = kb_total;
    if (!encode_tmap_3d(&p.tmap_a[s], es, d->a_ptr[s], (uint64_t)d->a_channels[s], (uint64_t)d->a_rows_per_utt[s],
                        (uint64_t)d->B, (uint64_t)d->a_ld[s] * es,
                        (uint64_t)d->a_rows_per_utt[s] * (uint64_t)d->a_ld[s] * es, kc, tb, p.bb))
      return -3;
  }
  p.num_kb = kb_total;
  AVC_REQUIRE(kb_total * kc == d->k_pad, "avc_conv_gemm: k_pad %d != %d k-blocks x %d", d->k_pad, kb_total, kc);
  const long long m_tiles = (long long)p.tiles_t * tiles_b;
  int ctas = d->cta_group == 1 ? 1 : 2;     // CTA pairs unless the descriptor asks for single CTAs
  if (m_tiles < 2) ctas = 1;
  // each CTA of a pair stages bn / 2 rows of the weight tile
  if (!encode_tmap_2d(&p.tmap_b, es, d->w_ptr, (uint64_t)d->k_pad, (uint64_t)d->n_pad, (uint64_t)d->k_pad * es, kc,
                      bn / ctas))
    return -3;

  p.bias = d->bias;
  p.act = d->act;
  p.phases = d->out_phases > 0 ? d->out_phases : 1;
  // a launch may produce only `out_phase_count` consecutive phases starting at `out_phase0` (the two halves of a
  // ConvTranspose1d use different pairs of input taps and run as two GEMMs without the all-zero third tap)
  const int phase_count = d->out_phase_count > 0 ? d->out_phase_count : p.phases;
  p.phase0 = d->out_phase0;
  AVC_REQUIRE(p.phase0 >= 0 && p.phase0 + phase_count <= p.phases, "avc_conv_gemm: phases [%d, %d) of %d", p.phase0,
              p.phase0 + phase_count, p.phases);
  AVC_REQUIRE(d->N % phase_count == 0 && (d->N / phase_count) % 4 == 0, "avc_conv_gemm: N=%d not divisible into %d phases",
              d->N, phase_count);
  p.cs = d->N / phase_count;
  const long long t_out = (long long)d->T * p.phases;
  p.out = d->out;
  p.out_ld = d->out_ld;
  p.out_rows_per_utt = d->out_rows_per_utt;
  p.out_row0 = d->out_row0;
  p.out_mode = d->out_dtype;
  AVC_REQUIRE(d->out_dtype >= 0 && d->out_dtype <= 4, "avc_conv_gemm: out_dtype %d", d->out_dtype);
  // out_raw_dtype = 0 keeps the historical meaning "same format as out" (fp32 raw copies go through out2)
  p.raw_mode = d->out_raw_dtype > 0 ? d->out_raw_dtype : d->out_dtype;
  AVC_REQUIRE(p.raw_mode >= 0 && p.raw_mode <= 4, "avc_conv_gemm: out_raw_dtype %d", d->out_raw_dtype);
  p.fmt_xor = d->dtype == AVC_DTYPE_F16 ? kIdescF16Xor : 0u;
  const long long min_ld = (d->out_dtype == 2 || d->out_dtype == 4) ? 2LL * p.cs : p.cs;
  const long long min_raw_ld = (p.raw_mode == 2 || p.raw_mode == 4) ? 2LL * p.cs : p.cs;
  p.out_round = d->out_round_tf32;
  p.out_reflect = d->out_reflect;
  p.out_raw = d->out_raw;
  p.out_raw_ld = d->out_raw_ld;
  p.out2 = d->out2;
  p.out2_ld = d->out2_ld;
  p.residual = d->residual;
  p.res_ld = d->res_ld;
  p.res_after = d->res_after_act;
  p.debug_clk = d->debug_clk;
  if (d->out) {
    AVC_REQUIRE(d->out_ld % 4 == 0 && d->out_ld >= min_ld &&
                    d->out_rows_per_utt >= d->out_row0 + t_out + d->out_reflect && d->out_row0 >= d->out_reflect,
                "avc_conv_gemm: bad output geometry");
    AVC_REQUIRE(d->out_reflect < t_out, "avc_conv_gemm: reflect %d needs more than that many output frames",
                d->out_reflect);
  }
  if (d->out_raw) AVC_REQUIRE(d->out_raw_ld % 4 == 0 && d->out_raw_ld >= min_raw_ld, "avc_conv_gemm: out_raw_ld");
  if (d->out2) AVC_REQUIRE(d->out2_ld % 4 == 0 && d->out2_ld >= p.cs, "avc_conv_gemm: out2_ld");
  if (d->residual) AVC_REQUIRE(d->res_ld % 4 == 0 && d->res_ld >= p.cs, "avc_conv_gemm: res_ld");

  const bool bf16 = d->dtype != AVC_DTYPE_TF32;      // 16-bit operands (bf16 or fp16)
  switch (bn) {
    case 64: return bf16 ? launch<64, true>(p, m_tiles, ctas, stream) : launch<64, false>(p, m_tiles, ctas, stream);
    case 128: return bf16 ? launch<128, true>(p, m_tiles, ctas, stream) : launch<128, false>(p, m_tiles, ctas, stream);
    default: return bf16 ? launch<256, true>(p, m_tiles, ctas, stream) : launch<256, false>(p, m_tiles, ctas, stream);
  }
}
