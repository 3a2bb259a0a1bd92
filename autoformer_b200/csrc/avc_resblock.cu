// Fused MelGAN ResnetBlock for the narrow, long stages (C = 32 / 64 channels), split-bf16 precision
// (see include/avc_b200.h: avc_resblock; melgan/modules.py:72-85).
//
//   y = W_sc x + W_1 LeakyReLU( W_3 *_d LeakyReLU(x) + b_3 ) + (b_1 + b_sc)
//
// Run layer by layer these blocks are bound by HBM and by bytes in flight: the dilated k3 convolution re-loads
// every activation row once per tap and per split-precision term (9 k-blocks of 16 KB per 128-row tile, of which
// 2 are new data), and the intermediate makes a round trip through HBM.  Here one CTA owns a tile of 128 output
// samples of one utterance and
//   * keeps all five weight matrices of the block resident in shared memory (80 KB for C = 64),
//   * loads ONE window of 128 + 2d rows of LeakyReLU(x); the three taps are the same shared-memory tile read through
//     operand descriptors whose start address is advanced by d rows (the 128-byte swizzle is a function of the
//     absolute shared-memory address, so a row-shifted descriptor stays consistent: scripts/ubench/desc_shift.cu),
//   * runs conv k3 -> TMEM -> (bias, LeakyReLU, hi/lo split) -> shared memory -> k1 + shortcut GEMM -> TMEM, so the
//     intermediate never leaves the SM,
//   * writes y / LeakyReLU(y) with TMA stores from swizzled staging tiles (full 128-byte rows).
// HBM traffic per block: read LeakyReLU(x) + x, write y + LeakyReLU(y) -- 4 tensor passes instead of 6, and every
// byte a CTA has in flight is new data.
//
// Split-bf16 products (DESIGN.md section 2) with one MMA per operand tile:
//   C = 64: activation tiles a_hi, a_lo (128 B rows); weight tile rows [W_hi (64) ; W_lo (64)]:
//           a_hi x tile (N = 128) -> D[0:64] = hi*hi, D[64:128] = hi*lo;  a_lo x tile[0:64] (N = 64) -> D[0:64] += lo*hi
//   C = 32: one activation tile whose 128-byte rows are [a_hi (32) | a_lo (32)]; weight tile rows
//           [ [W_hi | W_hi] (32) ; [W_lo | 0] (32) ]:  a x tile (N = 64) -> D[0:32] = hi*hi + lo*hi, D[32:64] = hi*lo
// and in both cases z[c] = D[c] + D[C + c].
//
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2..9 = epilogue (two warps per TMEM lane quarter, half of the
// channels each).  Per tile: GEMM1 -> epilogue 1 (intermediate to shared memory) -> GEMM2 -> epilogue 2 (stores);
// the window and x tiles of tile i+1 are loaded as soon as GEMM1 / GEMM2 of tile i have consumed theirs, and GEMM1 of
// tile i+1 runs under epilogue 2 of tile i.  C = 32 runs two CTAs per SM.
#include <cuda_bf16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

template <int C>
struct RbCfg {
  static_assert(C == 32 || C == 64, "fused ResnetBlock: 32 or 64 channels");
  static constexpr int kParts = C == 64 ? 2 : 1;              // operand tiles per block of rows
  static constexpr int kMaxDilation = 16;
  static constexpr int kWinTile = (kBlockM + 2 * kMaxDilation) * kRowBytes;   // 20 KB
  static constexpr int kWTile = 2 * C * kRowBytes;
  static constexpr int kOffW = 0;                              // W3 tap 0..2, W1, Wsc
  static constexpr int kOffWin = kOffW + 5 * kWTile;
  static constexpr int kOffXr = kOffWin + kParts * kWinTile;
  static constexpr int kOffMid = kOffXr + kParts * kATileBytes;
  static constexpr int kOffStage = kOffMid + kParts * kATileBytes;     // 128 rows x C x 4 bytes
  static constexpr int kOffBias = kOffStage + kParts * kATileBytes;
  static constexpr int kOffBar = kOffBias + 1024;
  static constexpr int kSmemBytes = kOffBar + 128 + 1024 /* alignment slack */;
  static constexpr uint32_t kTmemCols = 4 * C;                 // D1 and D2, 2C columns each
  static constexpr int kCtasPerSm = C == 32 ? 2 : 1;
  static_assert(kSmemBytes * kCtasPerSm + 1024 * kCtasPerSm <= 228 * 1024, "shared memory budget exceeded");
};

constexpr int kRbThreads = 64 + 32 * kEpiWarps;

struct alignas(64) RbParams {
  CUtensorMap tmap_win[2];    // LeakyReLU(x) with halo rows, (64, L + 2d, B) bf16, box {64, 128 + 2d, 1}
  CUtensorMap tmap_xr[2];     // x, (64, L, B), box {64, 128, 1}
  CUtensorMap tmap_out[2];    // LeakyReLU(y), operand format
  CUtensorMap tmap_raw[2];    // y, operand format
  CUtensorMap tmap_out2[2];   // LeakyReLU(y), fp32 (32, B * L), box {32, 128}
  const uint4* w;             // [5][2C][8 x 16 B]
  const float* bias3;
  const float* bias1;
  __nv_bfloat16* out;
  long long out_ld;
  int out_rows_per_utt, out_row0, out_reflect;
  int has_out, has_raw, has_out2;
  int B, L, dilation;
  int n_tiles, tiles_per_utt;
};

__device__ __forceinline__ void tma_store_3d(const void* tmap, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the committed stores have finished READING shared memory (the tiles may be overwritten)
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epilogue_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory"); }

// z[e] = D[col + e] + D[col + C + e] for NCH consecutive channels of the accumulator row this thread owns.
template <int C, int NCH>
__device__ __forceinline__ void load_sum(uint32_t taddr, float (&z)[NCH]) {
  uint32_t a[NCH], b[NCH];
  if constexpr (NCH == 32) {
    tmem_ld_32x32(taddr, a);
    tmem_ld_32x32(taddr + C, b);
  } else {
    tmem_ld_32x16(taddr, a);
    tmem_ld_32x16(taddr + C, b);
  }
  tmem_ld_wait();
#pragma unroll
  for (int e = 0; e < NCH; ++e) z[e] = __uint_as_float(a[e]) + __uint_as_float(b[e]);
}

// The MMAs of one activation source (tiles a0 [, a1]) against one weight tile.
template <int C>
__device__ __forceinline__ void issue_src(uint32_t a0, uint32_t a1, uint32_t w, uint32_t d, bool first) {
  if (C == 64) {
    constexpr uint32_t wide = umma_idesc(kBlockM, 128, false), narrow = umma_idesc(kBlockM, 64, false);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(d, umma_desc_sw128(a0 + k * 32), umma_desc_sw128(w + k * 32), wide, (first && k == 0) ? 0u : 1u);
#pragma unroll
    for (int k = 0; k < 4; ++k) umma_bf16(d, umma_desc_sw128(a1 + k * 32), umma_desc_sw128(w + k * 32), narrow, 1u);
  } else {
    constexpr uint32_t idesc = umma_idesc(kBlockM, 64, false);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(d, umma_desc_sw128(a0 + k * 32), umma_desc_sw128(w + k * 32), idesc, (first && k == 0) ? 0u : 1u);
  }
}

// slope < 1: LeakyReLU(v) = max(v, slope * v)
__device__ __forceinline__ float lrelu(float v) { return fmaxf(v, 0.2f * v); }

// Writes NCH channels starting at channel c0 of row `row` as split bf16 into operand tile(s) at `tiles`
// (C = 64: hi tile, lo tile; C = 32: one tile with [hi | lo] rows), 128-byte swizzle.
template <int C, int NCH>
__device__ __forceinline__ void write_split(uint8_t* tiles, int row, int c0, const float (&v)[NCH], uint4 (&hi)[NCH / 8],
                                            uint4 (&lo)[NCH / 8]) {
#pragma unroll
  for (int j = 0; j < NCH / 8; ++j) {
    float l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) l[e] = v[j * 8 + e] - __bfloat162float(__float2bfloat16_rn(v[j * 8 + e]));
    hi[j] = make_uint4(pack_bf16(v[j * 8], v[j * 8 + 1]), pack_bf16(v[j * 8 + 2], v[j * 8 + 3]),
                       pack_bf16(v[j * 8 + 4], v[j * 8 + 5]), pack_bf16(v[j * 8 + 6], v[j * 8 + 7]));
    lo[j] = make_uint4(pack_bf16(l[0], l[1]), pack_bf16(l[2], l[3]), pack_bf16(l[4], l[5]), pack_bf16(l[6], l[7]));
    const int chunk = c0 / 8 + j;
    uint8_t* r = tiles + row * kRowBytes;
    if (C == 64) {
      *reinterpret_cast<uint4*>(r + ((chunk ^ (row & 7)) << 4)) = hi[j];
      *reinterpret_cast<uint4*>(r + kATileBytes + ((chunk ^ (row & 7)) << 4)) = lo[j];
    } else {
      *reinterpret_cast<uint4*>(r + ((chunk ^ (row & 7)) << 4)) = hi[j];
      *reinterpret_cast<uint4*>(r + (((chunk + 4) ^ (row & 7)) << 4)) = lo[j];
    }
  }
}

template <int C>
__global__ void __launch_bounds__(kRbThreads, RbCfg<C>::kCtasPerSm) resblock_kernel(const __grid_constant__ RbParams p) {
  using Cfg = RbCfg<C>;
  constexpr int P = Cfg::kParts;
  constexpr int NCH = C / 2;                 // channels per epilogue thread
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_w = base + Cfg::kOffW;
  uint8_t* s_win = base + Cfg::kOffWin;
  uint8_t* s_xr = base + Cfg::kOffXr;
  uint8_t* s_mid = base + Cfg::kOffMid;
  uint8_t* s_stage = base + Cfg::kOffStage;
  float* s_bias = reinterpret_cast<float*>(base + Cfg::kOffBias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + Cfg::kOffBar);
  uint64_t* win_full = bars + 0;
  uint64_t* xr_full = bars + 1;
  uint64_t* d1_full = bars + 2;      // GEMM1 done: accumulator 1 ready, window tile free
  uint64_t* d2_full = bars + 3;      // GEMM2 done: accumulator 2 ready, x and intermediate tiles free
  uint64_t* mid_ready = bars + 4;    // intermediate written (and accumulator 1 drained) by all epilogue warps
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int win_rows = kBlockM + 2 * p.dilation;

  if (threadIdx.x == 0) {
    mbar_init(win_full, 1);
    mbar_init(xr_full, 1);
    mbar_init(d1_full, 1);
    mbar_init(d2_full, 1);
    mbar_init(mid_ready, kEpiWarps);
    fence_mbar_init();
#pragma unroll
    for (int part = 0; part < P; ++part) {
      prefetch_tmap(&p.tmap_win[part]);
      prefetch_tmap(&p.tmap_xr[part]);
    }
  }
  // weight tiles -> shared memory, 128-byte swizzle (row n, 16-byte chunk c at n * 128 + ((c ^ n % 8) << 4))
  for (int i = threadIdx.x; i < 5 * 2 * C * 8; i += kRbThreads) {
    const int n = i >> 3, c = i & 7;         // n runs over the rows of all five tiles (tiles are contiguous)
    *reinterpret_cast<uint4*>(s_w + n * kRowBytes + ((c ^ (n & 7)) << 4)) = p.w[i];
  }
  for (int i = threadIdx.x; i < 2 * C; i += kRbThreads) s_bias[i] = i < C ? p.bias3[i] : p.bias1[i - C];
  fence_proxy_async();          // the tensor core reads the weight tiles through the async proxy
  if (warp == 1) {
    tmem_alloc(tmem_ptr, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
  const uint32_t d1 = tmem_base, d2 = tmem_base + 2 * C;

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
        const int b = tile / p.tiles_per_utt, t0 = (tile % p.tiles_per_utt) * kBlockM;
        if (it > 0) mbar_wait(d1_full, (it - 1) & 1);
        mbar_arrive_expect_tx(win_full, P * win_rows * kRowBytes);
#pragma unroll
        for (int part = 0; part < P; ++part)
          tma_load_3d(s_win + part * Cfg::kWinTile, &p.tmap_win[part], win_full, 0, t0, b);
        if (it > 0) mbar_wait(d2_full, (it - 1) & 1);
        mbar_arrive_expect_tx(xr_full, P * kATileBytes);
#pragma unroll
        for (int part = 0; part < P; ++part)
          tma_load_3d(s_xr + part * kATileBytes, &p.tmap_xr[part], xr_full, 0, t0, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t w = smem_u32(s_w), win = smem_u32(s_win), xr = smem_u32(s_xr), mid = smem_u32(s_mid);
      const uint32_t shift = p.dilation * kRowBytes;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
        mbar_wait(win_full, it & 1);
        tc_fence_after();
#pragma unroll
        for (int tap = 0; tap < 3; ++tap)
          issue_src<C>(win + tap * shift, win + Cfg::kWinTile + tap * shift, w + tap * Cfg::kWTile, d1, tap == 0);
        umma_commit(d1_full);
        mbar_wait(mid_ready, it & 1);
        mbar_wait(xr_full, it & 1);
        tc_fence_after();
        issue_src<C>(mid, mid + kATileBytes, w + 3 * Cfg::kWTile, d2, true);
        issue_src<C>(xr, xr + kATileBytes, w + 4 * Cfg::kWTile, d2, false);
        umma_commit(d2_full);
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3;                    // TMEM lane quarter this warp may read
    const int h = (warp - 2) >> 2;             // which half of the channels
    const int row = q * 32 + lane;
    const int c0 = h * NCH;
    const uint32_t lane_addr = (static_cast<uint32_t>(q * 32) << 16) + c0;
    const bool storer = threadIdx.x == 64;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int b = tile / p.tiles_per_utt, t0 = (tile % p.tiles_per_utt) * kBlockM;
      float v[NCH];
      uint4 hi[NCH / 8], lo[NCH / 8];
      // ---- epilogue 1: intermediate = LeakyReLU(conv3 + b3) as an operand tile in shared memory
      mbar_wait(d1_full, it & 1);
      tc_fence_after();
      load_sum<C, NCH>(d1 + lane_addr, v);
#pragma unroll
      for (int e = 0; e < NCH; ++e) v[e] = lrelu(v[e] + s_bias[c0 + e]);
      if (it > 0) {          // the previous tile's TMA stores must have read the staging tiles (mid, stage)
        if (storer) bulk_wait_read();
        epilogue_bar();
      }
      write_split<C, NCH>(s_mid, row, c0, v, hi, lo);
      fence_proxy_async();   // generic-proxy writes -> tensor-core (async proxy) reads
      tc_fence_before();     // ... and this warp's reads of accumulator 1 before the next GEMM1
      __syncwarp();
      if (lane == 0) mbar_arrive(mid_ready);
      // ---- epilogue 2: y = k1(mid) + shortcut(x) + bias; stores
      mbar_wait(d2_full, it & 1);
      tc_fence_after();
      load_sum<C, NCH>(d2 + lane_addr, v);
#pragma unroll
      for (int e = 0; e < NCH; ++e) v[e] += s_bias[C + c0 + e];
      if (p.has_raw) write_split<C, NCH>(s_mid, row, c0, v, hi, lo);      // GEMM2 has consumed the intermediate
#pragma unroll
      for (int e = 0; e < NCH; ++e) v[e] = lrelu(v[e]);
      if (p.has_out) {
        write_split<C, NCH>(s_stage, row, c0, v, hi, lo);
        if (p.out_reflect > 0) {       // ReflectionPad1d rows of the consumer: time -k = time k, time L-1+k = time L-1-k
          const int t = t0 + row;
          int dst[2] = {-1, -1};
          if (t >= 1 && t <= p.out_reflect) dst[0] = p.out_row0 - t;
          if (t <= p.L - 2 && t >= p.L - 1 - p.out_reflect) dst[1] = p.out_row0 + 2 * (p.L - 1) - t;
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            if (dst[s] < 0) continue;
            __nv_bfloat16* o = p.out + ((long long)b * p.out_rows_per_utt + dst[s]) * p.out_ld + c0;
#pragma unroll
            for (int j = 0; j < NCH / 8; ++j) {
              *reinterpret_cast<uint4*>(o + j * 8) = hi[j];
              *reinterpret_cast<uint4*>(o + C + j * 8) = lo[j];
            }
          }
        }
      } else if (p.has_out2) {         // exact fp32 rows of 32 floats per 128-byte tile row
#pragma unroll
        for (int j = 0; j < NCH / 4; ++j) {
          const int f = c0 + j * 4;
          uint8_t* r = s_stage + (f >> 5) * kATileBytes + row * kRowBytes;
          *reinterpret_cast<float4*>(r + ((((f & 31) >> 2) ^ (row & 7)) << 4)) =
              make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
        }
      }
      fence_proxy_async();   // staging tiles -> TMA store (async proxy)
      tc_fence_before();
      epilogue_bar();
      if (storer) {
#pragma unroll
        for (int part = 0; part < P; ++part) {
          if (p.has_raw) tma_store_3d(&p.tmap_raw[part], s_mid + part * kATileBytes, 0, t0, b);
          if (p.has_out) tma_store_3d(&p.tmap_out[part], s_stage + part * kATileBytes, 0, p.out_row0 + t0, b);
          else if (p.has_out2) tma_store_2d(&p.tmap_out2[part], s_stage + part * kATileBytes, 0, b * p.L + t0);
        }
        bulk_commit();
      }
    }
    if (storer) bulk_wait_all();
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int C>
static int launch(const RbParams& p, cudaStream_t stream) {
  using Cfg = RbCfg<C>;
  auto kern = resblock_kernel<C>;
  static PerDeviceOnce configured;
  if (configured.first_use()) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  }
  const int max_ctas = num_sms() * Cfg::kCtasPerSm;
  const int grid = p.n_tiles < max_ctas ? p.n_tiles : max_ctas;
  kern<<<grid, kRbThreads, Cfg::kSmemBytes, stream>>>(p);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}


// =================================================================================================================
// Version 2 ("fp16s" precision, round 2): the block reads ONLY its raw input and writes ONLY its output.
//
// Version 1 above is bound by HBM: per block it reads LeakyReLU(x) and x and writes y and LeakyReLU(y) -- four tensor
// passes, because the activated copy of the residual stream exists as a tensor of its own.  Here the window of the raw
// residual stream x (two fp16 terms, reflected halo rows included) is the only input; the epilogue warps form the k3
// operand LeakyReLU(x) from it in shared memory (as ONE fp16 value: scripts/melgan_precision_study.py shows that operand
// tolerates it while the stream itself does not), and the shortcut GEMM reads the centre rows of the same window through
// a row-shifted descriptor.  Output: y (raw, with the next block's reflected halo) OR LeakyReLU(y) (the next
// ConvTranspose's operand) as two fp16 terms, or LeakyReLU(y) as exact fp32 -- one tensor.  Two passes instead of four.
//
//   x 2-term [hi | lo]  --TMA-->  window (double buffered)  --epilogue warps-->  xa = fp16(LeakyReLU(hi + lo))
//   GEMM1: D1 = sum_tap xa[rows + tap*d] . [W3_hi ; W3_lo]^T          (two products per tap: xa*w_hi + xa*w_lo)
//   mid   = LeakyReLU(D1 + b3) as two fp16 terms in shared memory
//   GEMM2: D2 = [mid_hi, mid_lo] . W1 + [x_hi, x_lo](centre rows) . Wsc   (three products each)
//
// (Tried and measured slower, r02: staging the output in the window buffer the tile has just finished with and letting
// the producer thread issue the TMA stores, so that no epilogue warp waits for a store -- the reload of that buffer for
// tile i+2 then starts a store later, the window's HBM latency is no longer covered by one tile period, and a block takes
// 0.73 ms (C = 64) / 0.68 ms (C = 32) instead of 0.60 ms.)
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2..9 = epilogue (two per TMEM lane quarter), 10..13 = xa warps.
// Schedule per CTA: the xa warps form xa(i+1) as soon as GEMM1(i) has read the xa tile, the epilogue warps run
// ep1(i) -> ep2(i), the MMA thread GEMM1(i) -> GEMM2(i): GEMM2(i) and ep1/ep2(i) overlap the xa pass of the next tile,
// GEMM1(i+1) overlaps ep2(i); the window of tile i+2 is loaded as soon as GEMM2(i) has read the centre rows of its buffer.
template <int C>
struct Rb2Cfg {
  static_assert(C == 32 || C == 64, "fused ResnetBlock: 32 or 64 channels");
  static constexpr int kParts = C == 64 ? 2 : 1;              // 128-byte-row tiles per block of rows (hi, lo | [hi|lo])
  static constexpr int kMaxDilation = 16;
  static constexpr int kWinTile = (kBlockM + 2 * kMaxDilation) * kRowBytes;   // 20 KB
  static constexpr int kW3Tile = (C == 64 ? 128 : 32) * kRowBytes;  // C=64: rows [w_hi(64); w_lo(64)]; C=32: rows [w_hi | w_lo]
  static constexpr int kW1Tile = (C == 64 ? 128 : 64) * kRowBytes;  // as version 1
  static constexpr int kOffW3 = 0;
  static constexpr int kOffW1 = kOffW3 + 3 * kW3Tile;
  static constexpr int kOffWsc = kOffW1 + kW1Tile;
  static constexpr int kWBytes = kOffWsc + kW1Tile;
  static constexpr int kOffWin = kWBytes;                              // two window buffers
  static constexpr int kOffXa = kOffWin + 2 * kParts * kWinTile;
  static constexpr int kOffMid = kOffXa + kWinTile;                    // intermediate, later the output staging tiles
  static constexpr int kOffBias = kOffMid + kParts * kATileBytes;
  // bias region: [0, 2C) the two bias vectors, [64, 64 + 7 * 32) the output convolution's taps
  static constexpr int kOffBar = kOffBias + 2048;
  static constexpr int kSmemBytes = kOffBar + 128 + 1024 /* alignment slack */;
  static constexpr uint32_t kD1Cols = C == 64 ? 128 : 32;
  static constexpr uint32_t kD2Cols = 2 * C;
  static constexpr uint32_t kTmemCols = C == 64 ? 256 : 128;
  static constexpr int kCtasPerSm = C == 32 ? 2 : 1;
  // epilogue warps: a multiple of 4 (one set per TMEM lane quarter).  16 warps for C = 64 (16 channels per thread) were
  // measured SLOWER than 8 (0.62 ms against 0.58 ms per block at B = 32, L = 128,000: the passes are bound by issue
  // slots, not by latency), so both widths run 8
  static constexpr int kEpi = 8;
  static constexpr int kThreads = 64 + 32 * kEpi + 32 * 4 /* xa warps */;
  static_assert(kWBytes % 1024 == 0 && kWinTile % 1024 == 0, "tiles must stay 1024-byte aligned");
  static_assert(kSmemBytes * kCtasPerSm + 1024 * kCtasPerSm <= 228 * 1024, "shared memory budget exceeded");
};

struct alignas(64) Rb2Params {
  CUtensorMap tmap_win[2];    // x with halo rows, (64, L + 2d, B) fp16, box {64, 128 + 2d, 1}; part p at channel 64 p
  CUtensorMap tmap_y[2];      // output (raw y or LeakyReLU(y)), two fp16 terms
  CUtensorMap tmap_out2[2];   // LeakyReLU(y), fp32 (32, B * L), box {32, 128}
  const uint4* w;             // packed tiles: W3 tap 0..2, W1, Wsc (packing.pack_resblock2)
  const float* bias3;
  const float* bias1;
  __half* y;
  long long y_ld;
  int y_rows_per_utt, y_row0, y_reflect, y_act;
  int has_y, has_out2;
  int B, L, dilation;
  int n_tiles, tiles_per_utt;
  // fused output convolution (C = 32): tiles overlap by K - 1 rows (tile_stride = 128 - (K - 1), the first row of a tile
  // is tile_lead = K / 2 samples before its first output) and only wav is written
  int tile_stride, tile_lead;
  const float* mono_w;        // [K][C] fp32
  float mono_bias;
  int mono_taps;
  float* wav;                 // [B][L] fp32
  // padded batch (RAGGED instantiation): valid rows per utterance and the prefix table of its tiles
  const int* lengths;
  const int* tile_start;
};

// Utterance and first window row of `tile`: fixed tiles_per_utt, or the compacted tile space of a padded batch.  Every
// role goes through here, so they all agree on the tile sequence and the ring / phase counting is unchanged.
template <bool RAGGED>
__device__ __forceinline__ void rb2_tile(const Rb2Params& p, int tile, int& b, int& t0) {
  if constexpr (RAGGED) {
    b = ragged_tile_utt(p.tile_start, p.B, tile);
    t0 = (tile - __ldg(p.tile_start + b)) * p.tile_stride - p.tile_lead;
  } else {
    b = tile / p.tiles_per_utt;
    t0 = (tile % p.tiles_per_utt) * p.tile_stride - p.tile_lead;
  }
}

// NCH channels starting at c0 of row `row` as two fp16 terms into operand tile(s) at `tiles`, 128-byte swizzle.
template <int C, int NCH>
__device__ __forceinline__ void write_split_f16(uint8_t* tiles, int row, int c0, const float (&v)[NCH], uint4 (&hi)[NCH / 8],
                                                uint4 (&lo)[NCH / 8]) {
#pragma unroll
  for (int j = 0; j < NCH / 8; ++j) {
    split_f16_pair_trunc(v[j * 8], v[j * 8 + 1], hi[j].x, lo[j].x);
    split_f16_pair_trunc(v[j * 8 + 2], v[j * 8 + 3], hi[j].y, lo[j].y);
    split_f16_pair_trunc(v[j * 8 + 4], v[j * 8 + 5], hi[j].z, lo[j].z);
    split_f16_pair_trunc(v[j * 8 + 6], v[j * 8 + 7], hi[j].w, lo[j].w);
    const int chunk = c0 / 8 + j;
    uint8_t* r = tiles + row * kRowBytes;
    if (C == 64) {
      *reinterpret_cast<uint4*>(r + ((chunk ^ (row & 7)) << 4)) = hi[j];
      *reinterpret_cast<uint4*>(r + kATileBytes + ((chunk ^ (row & 7)) << 4)) = lo[j];
    } else {
      *reinterpret_cast<uint4*>(r + ((chunk ^ (row & 7)) << 4)) = hi[j];
      *reinterpret_cast<uint4*>(r + (((chunk + 4) ^ (row & 7)) << 4)) = lo[j];
    }
  }
}

// xa = fp16(LeakyReLU(hi + lo)) for every row of the window, written with the window's own swizzle so that the three taps
// read it through row-shifted descriptors.  C = 32: rows [xa | xa] against weight rows [w_hi | w_lo].
constexpr int kXaWarps = 4;
template <int N>
__device__ __forceinline__ void epilogue_bar_n() { asm volatile("bar.sync 1, %0;" ::"n"(N) : "memory"); }

template <int C>
__device__ __forceinline__ void form_xa(const uint8_t* win, uint8_t* xa, int win_rows, int tid) {
  constexpr int CH = C / 8;                 // 16-byte chunks of one term per row
  for (int it = tid; it < win_rows * CH; it += 32 * kXaWarps) {
    const int r = it / CH, c = it - r * CH;
    const int sw = r & 7;
    const uint8_t* row = win + r * kRowBytes;
    const uint4 h = *reinterpret_cast<const uint4*>(row + ((c ^ sw) << 4));
    const uint4 l = C == 64 ? *reinterpret_cast<const uint4*>(row + Rb2Cfg<C>::kWinTile + ((c ^ sw) << 4))
                            : *reinterpret_cast<const uint4*>(row + (((c + 4) ^ sw) << 4));
    const __half2* hh = reinterpret_cast<const __half2*>(&h);
    const __half2* ll = reinterpret_cast<const __half2*>(&l);
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 a = __half22float2(hh[e]), b = __half22float2(ll[e]);
      o[e] = pack_f16(lrelu(a.x + b.x), lrelu(a.y + b.y));
    }
    const uint4 ov = make_uint4(o[0], o[1], o[2], o[3]);
    uint8_t* orow = xa + r * kRowBytes;
    *reinterpret_cast<uint4*>(orow + ((c ^ sw) << 4)) = ov;
    if (C == 32) *reinterpret_cast<uint4*>(orow + (((c + 4) ^ sw) << 4)) = ov;
  }
}

constexpr uint32_t idesc_f16(uint32_t n) { return umma_idesc(kBlockM, n, false) ^ kIdescF16Xor; }

// GEMM1: the three taps of the dilated convolution off the xa window.
template <int C>
__device__ __forceinline__ void issue_k3(uint32_t xa, uint32_t w3, uint32_t shift, uint32_t d1) {
  constexpr uint32_t idesc = idesc_f16(Rb2Cfg<C>::kD1Cols);
#pragma unroll
  for (int tap = 0; tap < 3; ++tap)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(d1, umma_desc_sw128(xa + tap * shift + k * 32), umma_desc_sw128(w3 + tap * Rb2Cfg<C>::kW3Tile + k * 32), idesc,
                (tap == 0 && k == 0) ? 0u : 1u);
}

// One two-term activation source (tiles a0 [, a1]) against one [w_hi ; w_lo]-style weight tile: three products.
template <int C>
__device__ __forceinline__ void issue_src_f16(uint32_t a0, uint32_t a1, uint32_t w, uint32_t d, bool first) {
  if (C == 64) {
    constexpr uint32_t wide = idesc_f16(128), narrow = idesc_f16(64);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(d, umma_desc_sw128(a0 + k * 32), umma_desc_sw128(w + k * 32), wide, (first && k == 0) ? 0u : 1u);
#pragma unroll
    for (int k = 0; k < 4; ++k) umma_bf16(d, umma_desc_sw128(a1 + k * 32), umma_desc_sw128(w + k * 32), narrow, 1u);
  } else {
    constexpr uint32_t idesc = idesc_f16(64);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(d, umma_desc_sw128(a0 + k * 32), umma_desc_sw128(w + k * 32), idesc, (first && k == 0) ? 0u : 1u);
  }
}

// RAGGED: a padded batch, only the tiles that hold a valid row (see avc_resblock2_desc.lengths).  A separate
// instantiation: the fixed-length one is compiled exactly as it is without lengths.
template <int C, bool RAGGED>
__global__ void __launch_bounds__(Rb2Cfg<C>::kThreads, Rb2Cfg<C>::kCtasPerSm) resblock2_kernel(const __grid_constant__ Rb2Params p) {
  using Cfg = Rb2Cfg<C>;
  constexpr int P = Cfg::kParts;
  constexpr int kEpi = Cfg::kEpi;
  constexpr int kThreads = Cfg::kThreads;
  constexpr int NCH = C / (kEpi / 4);        // channels per epilogue thread
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_w = base;
  uint8_t* s_win = base + Cfg::kOffWin;
  uint8_t* s_xa = base + Cfg::kOffXa;
  uint8_t* s_mid = base + Cfg::kOffMid;
  float* s_bias = reinterpret_cast<float*>(base + Cfg::kOffBias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + Cfg::kOffBar);
  uint64_t* win_full = bars + 0;     // [2] TMA bytes of a window buffer have landed
  uint64_t* win_free = bars + 2;     // [2] GEMM2 has read the centre rows of a window buffer (and xa was formed from it)
  uint64_t* xa_ready = bars + 4;     // xa tile written by all epilogue warps
  uint64_t* d1_full = bars + 5;      // GEMM1 done: accumulator 1 ready, xa tile free
  uint64_t* mid_ready = bars + 6;    // intermediate written (and accumulator 1 drained) by all epilogue warps
  uint64_t* d2_full = bars + 7;      // GEMM2 done: accumulator 2 ready, intermediate tiles free
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int win_rows = kBlockM + 2 * p.dilation;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&win_full[i], 1);
      mbar_init(&win_free[i], 1);
    }
    mbar_init(xa_ready, kXaWarps);
    mbar_init(d1_full, 1);
    mbar_init(mid_ready, kEpi);
    mbar_init(d2_full, 1);
    fence_mbar_init();
#pragma unroll
    for (int part = 0; part < P; ++part) prefetch_tmap(&p.tmap_win[part]);
  }
  // weight tiles -> shared memory, 128-byte swizzle (row n, 16-byte chunk c at n * 128 + ((c ^ n % 8) << 4)); every tile
  // starts on a multiple of 8 rows, so the global row index gives the right swizzle phase
  for (int i = threadIdx.x; i < Cfg::kWBytes / 16; i += kThreads) {
    const int n = i >> 3, c = i & 7;
    *reinterpret_cast<uint4*>(s_w + n * kRowBytes + ((c ^ (n & 7)) << 4)) = p.w[i];
  }
  for (int i = threadIdx.x; i < 2 * C; i += kThreads) s_bias[i] = i < C ? p.bias3[i] : p.bias1[i - C];
  if (C == 32 && p.wav != nullptr)
    for (int i = threadIdx.x; i < p.mono_taps * C; i += kThreads) s_bias[64 + i] = p.mono_w[i];
  fence_proxy_async();          // the tensor core reads the weight tiles through the async proxy
  if (warp == 1) {
    tmem_alloc(tmem_ptr, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
  const uint32_t d1 = tmem_base, d2 = tmem_base + Cfg::kD1Cols;

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
        int b, t0;
        rb2_tile<RAGGED>(p, tile, b, t0);
        const int buf = it & 1, use = it >> 1;
        if (use > 0) mbar_wait(&win_free[buf], (use - 1) & 1);
        mbar_arrive_expect_tx(&win_full[buf], P * win_rows * kRowBytes);
#pragma unroll
        for (int part = 0; part < P; ++part)
          tma_load_3d(s_win + (buf * P + part) * Cfg::kWinTile, &p.tmap_win[part], &win_full[buf], 0, t0, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t w = smem_u32(s_w), xa = smem_u32(s_xa), mid = smem_u32(s_mid);
      const uint32_t shift = p.dilation * kRowBytes;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        const uint32_t xc = smem_u32(s_win + buf * P * Cfg::kWinTile) + shift;      // centre rows of the raw window
        mbar_wait(xa_ready, it & 1);
        tc_fence_after();
        issue_k3<C>(xa, w + Cfg::kOffW3, shift, d1);
        umma_commit(d1_full);
        mbar_wait(mid_ready, it & 1);
        tc_fence_after();
        issue_src_f16<C>(mid, mid + kATileBytes, w + Cfg::kOffW1, d2, true);
        issue_src_f16<C>(xc, xc + Cfg::kWinTile, w + Cfg::kOffWsc, d2, false);
        umma_commit(d2_full);
        umma_commit(&win_free[buf]);
      }
    }
    __syncwarp();
  } else if (warp >= 2 + kEpi) {
    // ---------------- xa warps: the k3 operand of tile i from its raw window, as soon as GEMM1(i-1) has read the xa tile
    const int tid = threadIdx.x - (64 + 32 * kEpi);
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&win_full[buf], (it >> 1) & 1);
      if (it > 0) mbar_wait(d1_full, (it - 1) & 1);
      form_xa<C>(s_win + buf * P * Cfg::kWinTile, s_xa, win_rows, tid);
      fence_proxy_async();   // generic-proxy writes -> tensor-core (async proxy) reads
      __syncwarp();
      if (lane == 0) mbar_arrive(xa_ready);
    }
  } else {
    const int q = warp & 3;                    // TMEM lane quarter this warp may read
    const int h = (warp - 2) >> 2;             // which half of the channels
    const int row = q * 32 + lane;
    const int c0 = h * NCH;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const bool storer = threadIdx.x == 64;
    const bool mono = C == 32 && p.wav != nullptr;
    float* const s_mono_w = s_bias + 64;
    float* const s_part = reinterpret_cast<float*>(s_mid);      // [2 channel halves][8][128] partial sums (8 KB of 16)
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      int b, t0;
      rb2_tile<RAGGED>(p, tile, b, t0);
      float v[NCH];
      uint4 hi[NCH / 8], lo[NCH / 8];
      // ---- epilogue 1: intermediate = LeakyReLU(conv3 + b3) as two fp16 terms in shared memory
      mbar_wait(d1_full, it & 1);
      tc_fence_after();
      if constexpr (C == 64) {
        load_sum<64, NCH>(d1 + lane_off + c0, v);          // D1 = [xa * w_hi (64) | xa * w_lo (64)]
      } else {
        uint32_t a[NCH];
        tmem_ld_32x16(d1 + lane_off + c0, a);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < NCH; ++e) v[e] = __uint_as_float(a[e]);
      }
#pragma unroll
      for (int e = 0; e < NCH; ++e) v[e] = lrelu(v[e] + s_bias[c0 + e]);
      if (it > 0) {          // the previous tile's TMA stores must have read the staging tiles (= the intermediate tiles)
        if (storer) bulk_wait_read();
        epilogue_bar_n<32 * kEpi>();
      }
      write_split_f16<C, NCH>(s_mid, row, c0, v, hi, lo);
      fence_proxy_async();   // generic-proxy writes -> tensor-core (async proxy) reads
      tc_fence_before();     // ... and this warp's reads of accumulator 1 before the next GEMM1
      __syncwarp();
      if (lane == 0) mbar_arrive(mid_ready);
      // ---- epilogue 2: y = k1(mid) + shortcut(x) + bias; store
      mbar_wait(d2_full, it & 1);
      tc_fence_after();
      load_sum<C, NCH>(d2 + lane_off + c0, v);
#pragma unroll
      for (int e = 0; e < NCH; ++e) v[e] += s_bias[C + c0 + e];
      if (p.y_act || p.has_out2 || mono) {
#pragma unroll
        for (int e = 0; e < NCH; ++e) v[e] = lrelu(v[e]);
      }
      if (p.has_y) {
        write_split_f16<C, NCH>(s_mid, row, c0, v, hi, lo);      // GEMM2 has consumed the intermediate
        if (p.y_reflect > 0) {         // ReflectionPad1d rows of the consumer: time -k = time k, time L-1+k = time L-1-k
          const int t = t0 + row;
          int dst[2] = {-1, -1};
          if (t >= 1 && t <= p.y_reflect) dst[0] = p.y_row0 - t;
          if (t <= p.L - 2 && t >= p.L - 1 - p.y_reflect) dst[1] = p.y_row0 + 2 * (p.L - 1) - t;
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            if (dst[s] < 0) continue;
            __half* o = p.y + ((long long)b * p.y_rows_per_utt + dst[s]) * p.y_ld + c0;
#pragma unroll
            for (int j = 0; j < NCH / 8; ++j) {
              *reinterpret_cast<uint4*>(o + j * 8) = hi[j];
              *reinterpret_cast<uint4*>(o + C + j * 8) = lo[j];
            }
          }
        }
      } else if (mono) {
        // the generator's output layer (melgan/modules.py:119-124: ReflectionPad1d(K/2), Conv1d(C -> 1, K), tanh) on this
        // thread's own row of LeakyReLU(y), still in registers: one partial dot product per tap over its 16 channels,
        // [channel half][tap][row] in the (now free) intermediate tile -- re-reading staged rows once per tap instead cost
        // 114 KB of shared-memory reads per tile (measured: 1.08 ms for the block against 0.62 ms un-fused)
        for (int k = 0; k < p.mono_taps; ++k) {
          const float4* wr = reinterpret_cast<const float4*>(s_mono_w + k * C + c0);
          float a0 = 0.f, a1 = 0.f;
#pragma unroll
          for (int j = 0; j < NCH / 4; ++j) {
            const float4 wv = wr[j];
            a0 = fmaf(v[j * 4], wv.x, a0);
            a1 = fmaf(v[j * 4 + 1], wv.y, a1);
            a0 = fmaf(v[j * 4 + 2], wv.z, a0);
            a1 = fmaf(v[j * 4 + 3], wv.w, a1);
          }
          s_part[(h * 8 + k) * kBlockM + row] = a0 + a1;
        }
      } else {                         // exact fp32 rows of 32 floats per 128-byte tile row
#pragma unroll
        for (int j = 0; j < NCH / 4; ++j) {
          const int f = c0 + j * 4;
          uint8_t* r = s_mid + (f >> 5) * kATileBytes + row * kRowBytes;
          *reinterpret_cast<float4*>(r + ((((f & 31) >> 2) ^ (row & 7)) << 4)) =
              make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
        }
      }
      fence_proxy_async();   // staging tiles -> TMA store (async proxy)
      tc_fence_before();
      epilogue_bar_n<32 * kEpi>();
      if constexpr (C == 32) {
        if (mono) {
          // output r of this tile is sample t0 + K/2 + r: the sum over the taps k of the per-row partial dot products of
          // tile rows r + k (mirrored at the two ends of the utterance), both channel halves
          const int K = p.mono_taps, t = t0 + p.tile_lead + row;
          const int len = RAGGED ? __ldg(p.lengths + b) : p.L;     // mirrored at the utterance's own last sample
          if (h == 0 && row < p.tile_stride && t < p.L) {
            if (RAGGED && t >= len) {
              p.wav[(long long)b * p.L + t] = 0.f;
            } else {
              float acc = p.mono_bias;
              for (int k = 0; k < K; ++k) {
                int tau = t + k - p.tile_lead;
                if (tau < 0) tau = -tau;
                if (tau >= len) tau = 2 * (len - 1) - tau;
                const int rr = tau - t0;
                acc += s_part[k * kBlockM + rr] + s_part[(8 + k) * kBlockM + rr];
              }
              p.wav[(long long)b * p.L + t] = tanh_fast(acc);
            }
          }
          continue;          // nothing is stored by TMA; the next tile's barrier orders these reads before its writes
        }
      }
      if (storer) {
#pragma unroll
        for (int part = 0; part < P; ++part) {
          if (p.has_y) tma_store_3d(&p.tmap_y[part], s_mid + part * kATileBytes, 0, p.y_row0 + t0, b);
          else tma_store_2d(&p.tmap_out2[part], s_mid + part * kATileBytes, 0, b * p.L + t0);
        }
        bulk_commit();
      }
    }
    if (storer) bulk_wait_all();
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int C, bool RAGGED>
static int launch2(const Rb2Params& p, cudaStream_t stream) {
  using Cfg = Rb2Cfg<C>;
  auto kern = resblock2_kernel<C, RAGGED>;
  static PerDeviceOnce configured;
  if (configured.first_use()) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  }
  const int max_ctas = num_sms() * Cfg::kCtasPerSm;
  const int grid = p.n_tiles < max_ctas ? p.n_tiles : max_ctas;
  kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, stream>>>(p);
  AVC_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int launch_resblock2_big(const avc_resblock2_desc* d, cudaStream_t stream);   // avc_resblock_big.cu (C = 128)

}  // namespace avc

extern "C" int avc_resblock2(const avc_resblock2_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_resblock2: null descriptor");
  AVC_REQUIRE(d->C == 32 || d->C == 64 || d->C == 128, "avc_resblock2: C=%d (32, 64 or 128)", d->C);
  AVC_REQUIRE(d->B > 0 && d->L > 0 && d->L % kBlockM == 0, "avc_resblock2: B=%d L=%d (L must be a multiple of 128)",
              d->B, d->L);
  AVC_REQUIRE(d->dilation >= 1 && d->dilation <= 16, "avc_resblock2: dilation %d (1..16)", d->dilation);
  AVC_REQUIRE(d->x && d->w && d->bias3 && d->bias1, "avc_resblock2: missing buffer");
  AVC_REQUIRE(d->x_ld >= 2 * d->C, "avc_resblock2: input row stride too small");
  AVC_REQUIRE((d->y != nullptr) + (d->out2 != nullptr) + (d->wav != nullptr) == 1,
              "avc_resblock2: exactly one of y / out2 / wav");
  AVC_REQUIRE(!d->wav || (d->C == 32 && d->mono_w && d->mono_taps % 2 == 1 && d->mono_taps >= 3 && d->mono_taps <= 7 &&
                          d->L > d->mono_taps),
              "avc_resblock2: the fused output convolution takes C = 32 and 3, 5 or 7 taps (C=%d, %d taps)", d->C,
              d->mono_taps);
  AVC_REQUIRE((long long)d->B * d->L < (1LL << 31), "avc_resblock2: B*L too large");
  if (d->lengths) {
    const int stride = d->wav ? kBlockM - (d->mono_taps - 1) : kBlockM;
    AVC_REQUIRE(d->tile_start && d->n_tiles >= d->B && d->n_tiles <= (long long)d->B * ((d->L + stride - 1) / stride),
                "avc_resblock2: lengths need tile_start and n_tiles in [B, B * ceil(L / %d)] (n_tiles %d)", stride,
                d->n_tiles);
  }
  if (d->C == 128) return launch_resblock2_big(d, stream);
  const int C = d->C, P = C == 64 ? 2 : 1;
  const uint64_t B = (uint64_t)d->B, L = (uint64_t)d->L;
  Rb2Params p;
  memset(&p, 0, sizeof(p));
  const uint64_t win_rows = L + 2 * d->dilation;
  for (int part = 0; part < P; ++part) {
    const __half* x = static_cast<const __half*>(d->x) + part * 64;
    if (!encode_tmap_3d(&p.tmap_win[part], 2, x, 64, win_rows, B, (uint64_t)d->x_ld * 2, win_rows * d->x_ld * 2, 64,
                        kBlockM + 2 * d->dilation, 1))
      return -3;
    if (d->y) {
      AVC_REQUIRE(d->y_ld >= 2 * C && d->y_row0 >= d->y_reflect && d->y_reflect >= 0 && d->y_reflect <= 16 &&
                      d->y_rows_per_utt >= d->y_row0 + d->L + d->y_reflect,
                  "avc_resblock2: bad y geometry (ld %lld rows %d row0 %d reflect %d)", d->y_ld, d->y_rows_per_utt,
                  d->y_row0, d->y_reflect);
      const __half* o = static_cast<const __half*>(d->y) + part * 64;
      if (!encode_tmap_3d(&p.tmap_y[part], 2, o, 64, (uint64_t)d->y_rows_per_utt, B, (uint64_t)d->y_ld * 2,
                          (uint64_t)d->y_rows_per_utt * d->y_ld * 2, 64, kBlockM, 1))
        return -3;
    }
    if (d->out2) {
      AVC_REQUIRE(d->out2_ld >= C, "avc_resblock2: out2_ld too small");
      if (!encode_tmap_2d(&p.tmap_out2[part], 4, d->out2 + part * 32, 32, B * L, (uint64_t)d->out2_ld * 4, 32, kBlockM))
        return -3;
    }
  }
  p.w = static_cast<const uint4*>(d->w);
  p.bias3 = d->bias3;
  p.bias1 = d->bias1;
  p.y = static_cast<__half*>(d->y);
  p.y_ld = d->y_ld;
  p.y_rows_per_utt = d->y_rows_per_utt;
  p.y_row0 = d->y_row0;
  p.y_reflect = d->y ? d->y_reflect : 0;
  p.y_act = d->y_act;
  p.has_y = d->y != nullptr;
  p.has_out2 = d->out2 != nullptr;
  p.B = d->B;
  p.L = d->L;
  p.dilation = d->dilation;
  p.tile_stride = kBlockM;
  p.tiles_per_utt = d->L / kBlockM;
  if (d->wav) {
    p.wav = d->wav;
    p.mono_w = d->mono_w;
    p.mono_bias = d->mono_bias;
    p.mono_taps = d->mono_taps;
    p.tile_lead = d->mono_taps / 2;
    p.tile_stride = kBlockM - (d->mono_taps - 1);
    p.tiles_per_utt = (d->L + p.tile_stride - 1) / p.tile_stride;
  }
  p.n_tiles = d->B * p.tiles_per_utt;
  if (d->lengths) {
    p.lengths = d->lengths;
    p.tile_start = d->tile_start;
    p.n_tiles = d->n_tiles;
    return C == 64 ? launch2<64, true>(p, stream) : launch2<32, true>(p, stream);
  }
  return C == 64 ? launch2<64, false>(p, stream) : launch2<32, false>(p, stream);
}

extern "C" int avc_resblock(const avc_resblock_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_resblock: null descriptor");
  AVC_REQUIRE(d->C == 32 || d->C == 64, "avc_resblock: C=%d (32 or 64)", d->C);
  AVC_REQUIRE(d->B > 0 && d->L > 0 && d->L % kBlockM == 0, "avc_resblock: B=%d L=%d (L must be a multiple of 128)",
              d->B, d->L);
  AVC_REQUIRE(d->dilation >= 1 && d->dilation <= 16, "avc_resblock: dilation %d (1..16)", d->dilation);
  AVC_REQUIRE(d->xa && d->x && d->w && d->bias3 && d->bias1, "avc_resblock: missing buffer");
  AVC_REQUIRE(d->xa_ld >= 2 * d->C && d->x_ld >= 2 * d->C, "avc_resblock: input row strides too small");
  AVC_REQUIRE(d->out || d->out_raw || d->out2, "avc_resblock: no output requested");
  AVC_REQUIRE(!(d->out && d->out2), "avc_resblock: out and out2 are exclusive");
  AVC_REQUIRE((long long)d->B * d->L < (1LL << 31), "avc_resblock: B*L too large");
  const int C = d->C, P = C == 64 ? 2 : 1;
  const uint64_t B = (uint64_t)d->B, L = (uint64_t)d->L;
  RbParams p;
  memset(&p, 0, sizeof(p));
  const uint64_t win_rows = L + 2 * d->dilation;
  for (int part = 0; part < P; ++part) {
    const __nv_bfloat16* xa = static_cast<const __nv_bfloat16*>(d->xa) + part * 64;
    const __nv_bfloat16* x = static_cast<const __nv_bfloat16*>(d->x) + part * 64;
    if (!encode_tmap_3d(&p.tmap_win[part], 2, xa, 64, win_rows, B, (uint64_t)d->xa_ld * 2, win_rows * d->xa_ld * 2, 64,
                        kBlockM + 2 * d->dilation, 1))
      return -3;
    if (!encode_tmap_3d(&p.tmap_xr[part], 2, x, 64, L, B, (uint64_t)d->x_ld * 2, L * d->x_ld * 2, 64, kBlockM, 1))
      return -3;
    if (d->out) {
      AVC_REQUIRE(d->out_ld >= 2 * C && d->out_row0 >= d->out_reflect && d->out_reflect >= 0 && d->out_reflect <= 16 &&
                      d->out_rows_per_utt >= d->out_row0 + d->L + d->out_reflect,
                  "avc_resblock: bad out geometry (ld %lld rows %d row0 %d reflect %d)", d->out_ld,
                  d->out_rows_per_utt, d->out_row0, d->out_reflect);
      const __nv_bfloat16* o = static_cast<const __nv_bfloat16*>(d->out) + part * 64;
      if (!encode_tmap_3d(&p.tmap_out[part], 2, o, 64, (uint64_t)d->out_rows_per_utt, B, (uint64_t)d->out_ld * 2,
                          (uint64_t)d->out_rows_per_utt * d->out_ld * 2, 64, kBlockM, 1))
        return -3;
    }
    if (d->out_raw) {
      AVC_REQUIRE(d->out_raw_ld >= 2 * C, "avc_resblock: out_raw_ld too small");
      const __nv_bfloat16* o = static_cast<const __nv_bfloat16*>(d->out_raw) + part * 64;
      if (!encode_tmap_3d(&p.tmap_raw[part], 2, o, 64, L, B, (uint64_t)d->out_raw_ld * 2, L * d->out_raw_ld * 2, 64,
                          kBlockM, 1))
        return -3;
    }
    if (d->out2) {
      AVC_REQUIRE(d->out2_ld >= C, "avc_resblock: out2_ld too small");
      if (!encode_tmap_2d(&p.tmap_out2[part], 4, d->out2 + part * 32, 32, B * L, (uint64_t)d->out2_ld * 4, 32, kBlockM))
        return -3;
    }
  }
  p.w = static_cast<const uint4*>(d->w);
  p.bias3 = d->bias3;
  p.bias1 = d->bias1;
  p.out = static_cast<__nv_bfloat16*>(d->out);
  p.out_ld = d->out_ld;
  p.out_rows_per_utt = d->out_rows_per_utt;
  p.out_row0 = d->out_row0;
  p.out_reflect = d->out ? d->out_reflect : 0;
  p.has_out = d->out != nullptr;
  p.has_raw = d->out_raw != nullptr;
  p.has_out2 = d->out2 != nullptr;
  p.B = d->B;
  p.L = d->L;
  p.dilation = d->dilation;
  p.tiles_per_utt = d->L / kBlockM;
  p.n_tiles = d->B * p.tiles_per_utt;
  return C == 64 ? launch<64>(p, stream) : launch<32>(p, stream);
}
