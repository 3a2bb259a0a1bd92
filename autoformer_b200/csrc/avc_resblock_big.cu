// Fused MelGAN ResnetBlock for the WIDE stage (C = 128), "fp16s" precision (see include/avc_b200.h: avc_resblock2;
// melgan/modules.py:72-85).  Same arithmetic and data flow as resblock2_kernel in avc_resblock.cu -- the block reads only
// the raw residual stream and writes only its output -- but five 128 x 128 two-term weight matrices are 320 KB and cannot
// stay in one SM's shared memory, so:
//   * a CTA PAIR (tcgen05 cta_group::2, M = 256) owns two 128-sample tiles; every weight tile is split over the pair
//     (CTA r stages rows [w_hi[64r..64r+64) ; w_lo[64r..64r+64)] of a 64-channel k-chunk), so each CTA streams 160 KB of
//     weights per tile out of L2 through a TMA ring -- 26 B/clk/SM -- while all MMAs are N = 256 wide (or N = 128 for the
//     a_lo * w_hi products), the width at which the tensor pipe, not the shared-memory port, sets the pace;
//   * the A operands never move: the raw window (two fp16 terms, 128 + 2d rows, loaded ONCE per tile), the k3 operand
//     xa = fp16(LeakyReLU(x)) formed from it in shared memory, and the intermediate (two fp16 terms) written by the
//     epilogue -- the three taps and the shortcut read the window / xa tiles through row-shifted descriptors.
// Layer by layer (avc_conv_gemm) the same block re-loads every activation row once per tap and per product out of L2
// (64 B/clk/SM: the L2 port, not the tensor pipe, bounds it) and round-trips the intermediate through HBM.
//
// Shared memory (single-buffered: 512 TMEM columns and 220 KB leave no room for a second set):
//   region A  76 KB  raw window [term][chunk] (128 + 2d rows x 128 B each)
//   region B  70 KB  [0, 38 KB) xa [chunk] (GEMM1's operand); [0, 64 KB) later the intermediate [term][chunk] (GEMM2's
//                    operand); [38 KB, 70 KB) the staging tiles of the TMA stores.  The output goes out in two passes, the hi
//                    terms then the lo terms of all 128 channels (32 KB each), so that staging and the NEXT tile's xa
//                    never overlap: xa is formed the moment the next window lands, while this tile is still being stored
//   ring      4 x 16 KB  weight tiles (this CTA's half)
// Per tile:  window load -> xa -> GEMM1 (3 taps x 2 chunks) -> epilogue 1 -> GEMM2 (k1 + shortcut, three products each)
// -> epilogue 2 -> TMA stores; the next window is requested as soon as GEMM2 has read the centre rows, and was
// prefetched into L2 while this tile computed.
// Warp roles: 0 = TMA producer, 1 = MMA issuer (leader CTA), 2..9 = epilogue, 10..17 = xa warps.
#include <cuda_fp16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

namespace big {

constexpr int C = 128;
constexpr int KC = C / 64;                        // 64-channel k-chunks
constexpr int kMaxDilation = 12;
constexpr int kWinRowsMax = kBlockM + 2 * kMaxDilation;          // 152
constexpr int kWinTile = kWinRowsMax * kRowBytes;                // 19 KB
constexpr int kBStage = 128 * kRowBytes;                         // this CTA's half of a weight tile: 16 KB
constexpr int kStages = 4;
constexpr int kOffWin = 0;
constexpr int kOffB = kOffWin + 2 * KC * kWinTile;               // region B
constexpr int kOffStage = KC * kWinTile;                         // staging tiles inside region B, behind the xa tiles
constexpr int kRegionB = kOffStage + KC * kATileBytes;           // 70 KB (the intermediate takes the first 64 KB)
constexpr int kOffRing = kOffB + kRegionB;
constexpr int kOffBias = kOffRing + kStages * kBStage;
constexpr int kOffBar = kOffBias + 2 * C * 4;
constexpr int kNumBars = 2 * kStages + 8;      // (7 used)
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024 /* alignment slack */;
constexpr int kXaWarps = 8;
constexpr int kThreads = 64 + 32 * kEpiWarps + 32 * kXaWarps;    // 576
constexpr int kStagesPerTile = 3 * KC + 2 * KC;                  // 10 weight tiles per 128-sample tile
static_assert(2 * KC * kATileBytes <= kRegionB, "the intermediate must fit region B");
static_assert(kWinTile % 1024 == 0 && kOffB % 1024 == 0 && kOffRing % 1024 == 0, "tiles must stay 1024-byte aligned");
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget exceeded");

struct alignas(64) Params {
  CUtensorMap tmap_x;      // x with halo rows, (2C, L + 2d, B) fp16, box {64, 128 + 2d, 1}
  CUtensorMap tmap_y;      // output, (2C, rows, B) fp16, box {64, 128, 1}
  CUtensorMap tmap_w;      // packed weights, (64, 5 * KC * 256) fp16, box {64, 128}
  const float* bias3;
  const float* bias1;
  __half* y;
  long long y_ld;
  int y_rows_per_utt, y_row0, y_reflect, y_act;
  int B, L, dilation;
  int n_tiles, tiles_per_utt, n_pairs;
  long long* debug_clk;    // optional: 16 clock64 stamps per tile of CTA 0 (first 64 tiles)
  const int* tile_start;   // RAGGED: [B + 1] prefix table of the tiles that hold a valid row (avc_resblock2_desc)
};

__device__ __forceinline__ void tma_store_3d(const void* tmap, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epilogue_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory"); }
__device__ __forceinline__ float lrelu(float v) { return fmaxf(v, 0.2f * v); }
constexpr uint32_t idesc2(uint32_t n) { return umma_idesc(2 * kBlockM, n, false) ^ kIdescF16Xor; }

// z[e] = D[col + e] + D[col + 64 + e], e < 32: the two column blocks of one output-channel group (see the kernel)
__device__ __forceinline__ void load_sum32(uint32_t taddr, float (&z)[32]) {
  uint32_t a[32], b[32];
  tmem_ld_32x32(taddr, a);
  tmem_ld_32x32(taddr + 64, b);
  tmem_ld_wait();
#pragma unroll
  for (int e = 0; e < 32; ++e) z[e] = __uint_as_float(a[e]) + __uint_as_float(b[e]);
}

// 32 channels starting at channel c0 of row `row` as two fp16 terms into the [term][chunk] operand tiles at `tiles`.
__device__ __forceinline__ void write_split32(uint8_t* tiles, int row, int c0, const float (&v)[32], uint4 (&hi)[4], uint4 (&lo)[4]) {
  uint8_t* r = tiles + (c0 >> 6) * kATileBytes + row * kRowBytes;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    split_f16_pair_trunc(v[j * 8], v[j * 8 + 1], hi[j].x, lo[j].x);
    split_f16_pair_trunc(v[j * 8 + 2], v[j * 8 + 3], hi[j].y, lo[j].y);
    split_f16_pair_trunc(v[j * 8 + 4], v[j * 8 + 5], hi[j].z, lo[j].z);
    split_f16_pair_trunc(v[j * 8 + 6], v[j * 8 + 7], hi[j].w, lo[j].w);
    const int chunk = ((c0 & 63) >> 3) + j;
    *reinterpret_cast<uint4*>(r + ((chunk ^ (row & 7)) << 4)) = hi[j];
    *reinterpret_cast<uint4*>(r + KC * kATileBytes + ((chunk ^ (row & 7)) << 4)) = lo[j];
  }
}

}  // namespace big

using namespace big;      // (the kernel itself lives in avc:: so that profilers list it beside the library's other kernels)

// RAGGED: a padded batch, only the tiles that hold a valid row; a separate instantiation, the fixed-length one is compiled
// exactly as it is without lengths.
template <bool RAGGED>
__global__ void __launch_bounds__(big::kThreads, 1) resblock2_big_kernel(const __grid_constant__ big::Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_win = base + kOffWin;         // [term][chunk] window tiles
  uint8_t* s_b = base + kOffB;             // xa [chunk] (kWinTile each) | mid / staging [term][chunk] (kATileBytes each)
  uint8_t* s_ring = base + kOffRing;
  float* s_bias = reinterpret_cast<float*>(base + kOffBias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + kOffBar);
  uint64_t* full = bars;                   // [kStages] weight tile landed (bytes of BOTH CTAs, on the leader's barrier)
  uint64_t* empty = bars + kStages;        // [kStages] the MMAs have read the stage (arrives in both CTAs)
  uint64_t* win_full = bars + 2 * kStages + 0;    // this CTA's window has landed
  uint64_t* xa_ready = bars + 2 * kStages + 1;    // leader: xa written by the xa warps of BOTH CTAs
  uint64_t* d1_full = bars + 2 * kStages + 2;     // GEMM1 done (both CTAs)
  uint64_t* mid_ready = bars + 2 * kStages + 3;   // leader: intermediate written by the epilogue warps of BOTH CTAs
  uint64_t* d2_full = bars + 2 * kStages + 4;     // GEMM2 done (both CTAs): window and intermediate are free
  uint64_t* d2_free = bars + 2 * kStages + 6;     // leader: the epilogue warps of BOTH CTAs have read accumulator 2
  uint64_t* win_free = bars + 2 * kStages + 5;    // the shortcut MMAs have read the window (both CTAs): it may be reloaded
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + kNumBars);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const bool leader = rank == 0;
  const int pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  const int win_rows = kBlockM + 2 * p.dilation;
  const uint32_t shift = p.dilation * kRowBytes;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(win_full, 1);
    mbar_init(xa_ready, 2 * kXaWarps);
    mbar_init(d1_full, 1);
    mbar_init(mid_ready, 2 * kEpiWarps);
    mbar_init(d2_full, 1);
    mbar_init(d2_free, 2 * kEpiWarps);
    mbar_init(win_free, 1);
    fence_mbar_init();
    prefetch_tmap(&p.tmap_x);
    prefetch_tmap(&p.tmap_w);
    prefetch_tmap(&p.tmap_y);
  }
  for (int i = threadIdx.x; i < 2 * C; i += kThreads) s_bias[i] = i < C ? p.bias3[i] : p.bias1[i - C];
  if (warp == 1) {
    tmem_alloc_2sm(tmem_ptr, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();        // the peer arrives on / credits bytes to the leader's barriers: inits must be visible cluster-wide
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
  const uint32_t d1 = tmem_base, d2 = tmem_base + 256;

  // profiling aid: stamp slot `k` of tile iteration `it` (CTA 0 only)
  auto stamp = [&](int it, int k) {
    if (p.debug_clk && blockIdx.x == 0 && it < 64) p.debug_clk[it * 16 + k] = clock64();
  };

  // tile of this CTA in pair-iteration `u`: 2u + rank (a phantom tile past the end loads zeros and stores nothing).  In a
  // padded batch the tiles are those that hold a valid row, and the two tiles of a pair may belong to two utterances.
  auto tile_coords = [&](int u, int& b, int& t0, bool& real) {
    const int tile = 2 * u + rank;
    real = tile < p.n_tiles;
    if constexpr (RAGGED) {
      b = p.B;                 // phantom: the utterance past the last one, all of it out of bounds
      t0 = 0;
      if (real) {
        b = ragged_tile_utt(p.tile_start, p.B, tile);
        t0 = (tile - __ldg(p.tile_start + b)) * kBlockM;
      }
    } else {
      b = tile / p.tiles_per_utt;
      t0 = (tile - b * p.tiles_per_utt) * kBlockM;
    }
  };

  if (warp == 0) {
    if (lane == 0) {
      RingState rs;
      int it = 0;
      for (int u = pair0; u < p.n_pairs; u += pair_stride, ++it) {
        int b, t0;
        bool real;
        tile_coords(u, b, t0, real);
        if (it > 0) mbar_wait(win_free, (it - 1) & 1);         // the previous tile's shortcut MMAs have read the window
        stamp(it, 0);                                          // window requested
        mbar_arrive_expect_tx(win_full, 2 * KC * win_rows * kRowBytes);
#pragma unroll
        for (int term = 0; term < 2; ++term)
#pragma unroll
          for (int kc = 0; kc < KC; ++kc)
            tma_load_3d(s_win + (term * KC + kc) * kWinTile, &p.tmap_x, win_full, term * C + kc * 64, t0, b);
        if (u + pair_stride < p.n_pairs) {                     // the next tile's window: into L2 while this one computes
          int nb, nt0;
          bool nreal;
          tile_coords(u + pair_stride, nb, nt0, nreal);
          if (nreal) {
#pragma unroll
            for (int i = 0; i < 2 * KC; ++i) tma_prefetch_3d(&p.tmap_x, i * 64, nt0, nb);
          }
        }
        for (int s = 0; s < kStagesPerTile; ++s) {             // weight tiles in CONSUMPTION order: W3 (tap, chunk), Wsc, W1
          // (packed order is W3, W1, Wsc: the shortcut is issued before k1, see the MMA thread)
          const int tile = s < 3 * KC ? s : (s < 4 * KC ? s + KC : s - KC);
          mbar_wait(&empty[rs.stage], rs.phase ^ 1u);
          if (leader) mbar_arrive_expect_tx(&full[rs.stage], 2 * kBStage);
          tma_load_2d_2sm(s_ring + rs.stage * kBStage, &p.tmap_w, &full[rs.stage], 0, tile * 256 + rank * 128);
          rs.advance<kStages>();
        }
        stamp(it, 1);                                          // all weight tiles of the tile requested
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      const uint32_t win = smem_u32(s_win), rb = smem_u32(s_b), ring = smem_u32(s_ring);
      RingState rs;
      int it = 0;
      for (int u = pair0; u < p.n_pairs; u += pair_stride, ++it) {
        // ---- GEMM1: D1 = sum_tap xa[rows + tap * d] . [w_hi | w_lo]^T, one N = 256 MMA per 16 channels
        mbar_spin_cluster(xa_ready, it & 1);
        stamp(it, 2);                                          // xa of both CTAs ready
        tc_fence_after();
        for (int tap = 0; tap < 3; ++tap) {
          for (int kc = 0; kc < KC; ++kc) {
            mbar_wait(&full[rs.stage], rs.phase);
            tc_fence_after();
            const uint32_t a = rb + kc * kWinTile + tap * shift, w = ring + rs.stage * kBStage;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_2sm(d1, umma_desc_sw128(a + k * 32), umma_desc_sw128(w + k * 32), idesc2(256),
                            (tap == 0 && kc == 0 && k == 0) ? 0u : 1u);
            umma_commit_2sm(&empty[rs.stage], 0x3);
            rs.advance<kStages>();
          }
        }
        umma_commit_2sm(d1_full, 0x3);
        stamp(it, 3);                                          // GEMM1 issued
        // ---- GEMM2: D2 = [x_hi, x_lo](centre rows) . Wsc + [mid_hi, mid_lo] . W1, three products per matrix:
        // a_hi . [w_hi | w_lo] (N = 256) and a_lo . w_hi (N = 128, landing on a column block of the same channels).
        // The shortcut half needs only the window, so it is issued right behind GEMM1 and runs while the epilogue warps
        // turn accumulator 1 into the intermediate; it must not overwrite accumulator 2 before the previous tile's
        // epilogue has read it.
        if (it > 0) mbar_spin_cluster(d2_free, (it - 1) & 1);
        tc_fence_after();
        for (int m = 0; m < 2; ++m) {
          if (m == 1) {
            umma_commit_2sm(win_free, 0x3);                    // GEMM1 (xa) and the shortcut (window) are the window's last readers
            mbar_spin_cluster(mid_ready, it & 1);
            stamp(it, 4);                                      // intermediate of both CTAs ready
            tc_fence_after();
          }
          for (int kc = 0; kc < KC; ++kc) {
            mbar_wait(&full[rs.stage], rs.phase);
            tc_fence_after();
            const uint32_t a_hi = m == 1 ? rb + kc * kATileBytes : win + kc * kWinTile + shift;
            const uint32_t a_lo = m == 1 ? a_hi + KC * kATileBytes : a_hi + KC * kWinTile;
            const uint32_t w = ring + rs.stage * kBStage;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_2sm(d2, umma_desc_sw128(a_hi + k * 32), umma_desc_sw128(w + k * 32), idesc2(256),
                            (m == 0 && kc == 0 && k == 0) ? 0u : 1u);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_2sm(d2 + 64, umma_desc_sw128(a_lo + k * 32), umma_desc_sw128(w + k * 32), idesc2(128), 1u);
            umma_commit_2sm(&empty[rs.stage], 0x3);
            rs.advance<kStages>();
          }
        }
        umma_commit_2sm(d2_full, 0x3);
        stamp(it, 5);                                          // GEMM2 issued
      }
    }
    __syncwarp();
  } else if (warp >= 2 + kEpiWarps) {
    // ---------------- xa warps: xa = fp16(LeakyReLU(hi + lo)) for every window row of both chunks
    const int tid = threadIdx.x - (64 + 32 * kEpiWarps);
    int it = 0;
    for (int u = pair0; u < p.n_pairs; u += pair_stride, ++it) {
      // (the window is requested as soon as the previous tile's shortcut MMAs have read the old one, i.e. while its k1
      // MMAs still run; the previous tile's staging tiles lie behind the xa tiles)
      mbar_wait(win_full, it & 1);
      if (tid == 0) stamp(it, 6);                               // window landed
      if (it > 0) mbar_wait(d2_full, (it - 1) & 1);             // ... and the intermediate under the xa tiles is dead
      // a warp takes 4 rows x 8 chunks per step; the (at most 5) steps of a chunk are unrolled so their shared-memory
      // loads and conversions overlap
      const int c = lane & 7, r0 = (warp - (2 + kEpiWarps)) * 4 + (lane >> 3);
#pragma unroll
      for (int kc = 0; kc < KC; ++kc) {
#pragma unroll
        for (int s = 0; s < (kWinRowsMax + 4 * kXaWarps - 1) / (4 * kXaWarps); ++s) {
          const int r = r0 + s * 4 * kXaWarps;
          if (r < win_rows) {
            const int off = r * kRowBytes + ((c ^ (r & 7)) << 4);
            const uint4 h = *reinterpret_cast<const uint4*>(s_win + kc * kWinTile + off);
            const uint4 l = *reinterpret_cast<const uint4*>(s_win + (KC + kc) * kWinTile + off);
            const __half2* hh = reinterpret_cast<const __half2*>(&h);
            const __half2* ll = reinterpret_cast<const __half2*>(&l);
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 a = __half22float2(hh[e]), bq = __half22float2(ll[e]);
              o[e] = pack_f16(lrelu(a.x + bq.x), lrelu(a.y + bq.y));
            }
            *reinterpret_cast<uint4*>(s_b + kc * kWinTile + off) = make_uint4(o[0], o[1], o[2], o[3]);
          }
        }
      }
      // generic-proxy writes -> tensor-core (async proxy) reads of THIS SM; the fence completes before the arrive below,
      // so a plain remote arrive is enough (a cluster-scope release would also drain every earlier global store)
      fence_proxy_async();
      __syncwarp();
      if (tid == 0) stamp(it, 8);                               // xa written (warp 0 of the xa warps)
      if (lane == 0) mbar_arrive_leader(xa_ready);
    }
  } else {
    // ---------------- epilogue warps: thread owns sample `row`; the two warps of a TMEM lane quarter take 64 channels each
    const int q = warp & 3;
    const int h = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const bool storer = threadIdx.x == 64;
    int it = 0;
    for (int u = pair0; u < p.n_pairs; u += pair_stride, ++it) {
      int b, t0;
      bool real;
      tile_coords(u, b, t0, real);
      float v[32];
      uint4 hi[4], lo[4];
      // accumulator columns of output channel c (both GEMMs): (c / 64) * 128 + c % 64 and the same + 64
      // ---- epilogue 1: intermediate = LeakyReLU(conv3 + b3), two fp16 terms, over the (dead) xa tiles
      mbar_wait(d1_full, it & 1);
      if (storer) stamp(it, 9);                                 // accumulator 1 ready
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < 2; ++sub) {
        const int c0 = h * 64 + sub * 32;
        load_sum32(d1 + lane_off + h * 128 + sub * 32, v);
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = lrelu(v[e] + s_bias[c0 + e]);
        write_split32(s_b, row, c0, v, hi, lo);
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (storer) stamp(it, 10);                                // intermediate written
      if (lane == 0) mbar_arrive_leader(mid_ready);
      // ---- epilogue 2: y = k1(mid) + shortcut(x) + bias, stored in two passes (hi terms, then lo terms) through the
      // 32 KB staging tiles; the accumulator is simply read twice
      mbar_wait(d2_full, it & 1);
      if (storer) stamp(it, 11);                                // accumulator 2 ready
      tc_fence_after();
#pragma unroll 1
      for (int term = 0; term < 2; ++term) {
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
          const int c0 = h * 64 + sub * 32;
          load_sum32(d2 + lane_off + h * 128 + sub * 32, v);
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] += s_bias[C + c0 + e];
          if (p.y_act) {
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = lrelu(v[e]);
          }
          uint4 part[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 hq, lq;
            split_f16_pair_trunc(v[j * 8], v[j * 8 + 1], hq.x, lq.x);
            split_f16_pair_trunc(v[j * 8 + 2], v[j * 8 + 3], hq.y, lq.y);
            split_f16_pair_trunc(v[j * 8 + 4], v[j * 8 + 5], hq.z, lq.z);
            split_f16_pair_trunc(v[j * 8 + 6], v[j * 8 + 7], hq.w, lq.w);
            part[j] = term == 0 ? hq : lq;
            const int chunk = ((c0 & 63) >> 3) + j;
            *reinterpret_cast<uint4*>(s_b + kOffStage + (c0 >> 6) * kATileBytes + row * kRowBytes +
                                      ((chunk ^ (row & 7)) << 4)) = part[j];
          }
          if (p.y_reflect > 0 && real) {   // ReflectionPad1d rows of the consumer: time -k = time k, time L-1+k = time L-1-k
            const int t = t0 + row;
            int dst[2] = {-1, -1};
            if (t >= 1 && t <= p.y_reflect) dst[0] = p.y_row0 - t;
            if (t <= p.L - 2 && t >= p.L - 1 - p.y_reflect) dst[1] = p.y_row0 + 2 * (p.L - 1) - t;
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              if (dst[s] < 0) continue;
              __half* o = p.y + ((long long)b * p.y_rows_per_utt + dst[s]) * p.y_ld + term * C + c0;
#pragma unroll
              for (int j = 0; j < 4; ++j) *reinterpret_cast<uint4*>(o + j * 8) = part[j];
            }
          }
        }
        if (term == 1) {       // this warp's reads of accumulator 2 are complete: the next tile's shortcut may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_leader(d2_free);
        }
        fence_proxy_async();   // staging tiles -> TMA store (async proxy)
        epilogue_bar();
        if (storer) {
          stamp(it, 12 + term);                                 // staging tiles of this pass written by all epilogue warps
          if (real) {
#pragma unroll
            for (int kc = 0; kc < KC; ++kc)
              tma_store_3d(&p.tmap_y, s_b + kOffStage + kc * kATileBytes, term * C + kc * 64, p.y_row0 + t0, b);
            bulk_commit();
            bulk_wait_read();
          }
        }
        epilogue_bar();        // the staging tiles are free again (for the next pass / the next tile's intermediate)
      }
    }
    if (storer) bulk_wait_all();
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();        // neither CTA may free TMEM / exit while the pair's MMAs or remote arrivals are pending
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

int launch_resblock2_big(const avc_resblock2_desc* d, cudaStream_t stream) {
  AVC_REQUIRE(d->C == C, "avc_resblock2: wide kernel is built for C = %d", C);
  AVC_REQUIRE(d->dilation <= kMaxDilation, "avc_resblock2: C = 128 supports dilation <= %d", kMaxDilation);
  AVC_REQUIRE(d->y != nullptr && d->out2 == nullptr, "avc_resblock2: C = 128 writes y only (two fp16 terms)");
  const uint64_t B = (uint64_t)d->B, L = (uint64_t)d->L;
  Params p;
  memset(&p, 0, sizeof(p));
  const uint64_t win_rows = L + 2 * d->dilation;
  if (!encode_tmap_3d(&p.tmap_x, 2, d->x, 2 * C, win_rows, B, (uint64_t)d->x_ld * 2, win_rows * d->x_ld * 2, 64,
                      kBlockM + 2 * d->dilation, 1))
    return -3;
  AVC_REQUIRE(d->y_ld >= 2 * C && d->y_row0 >= d->y_reflect && d->y_reflect >= 0 && d->y_reflect <= 16 &&
                  d->y_rows_per_utt >= d->y_row0 + d->L + d->y_reflect,
              "avc_resblock2: bad y geometry (ld %lld rows %d row0 %d reflect %d)", d->y_ld, d->y_rows_per_utt, d->y_row0,
              d->y_reflect);
  if (!encode_tmap_3d(&p.tmap_y, 2, d->y, 2 * C, (uint64_t)d->y_rows_per_utt, B, (uint64_t)d->y_ld * 2,
                      (uint64_t)d->y_rows_per_utt * d->y_ld * 2, 64, kBlockM, 1))
    return -3;
  if (!encode_tmap_2d(&p.tmap_w, 2, d->w, 64, (uint64_t)kStagesPerTile * 256, 128, 64, 128)) return -3;
  p.bias3 = d->bias3;
  p.bias1 = d->bias1;
  p.y = static_cast<__half*>(d->y);
  p.y_ld = d->y_ld;
  p.y_rows_per_utt = d->y_rows_per_utt;
  p.y_row0 = d->y_row0;
  p.y_reflect = d->y_reflect;
  p.y_act = d->y_act;
  p.B = d->B;
  p.L = d->L;
  p.dilation = d->dilation;
  p.tiles_per_utt = d->L / kBlockM;
  p.n_tiles = d->B * p.tiles_per_utt;
  if (d->lengths) {
    p.tile_start = d->tile_start;
    p.n_tiles = d->n_tiles;
  }
  p.n_pairs = (p.n_tiles + 1) / 2;
  p.debug_clk = d->debug_clk;
  auto kern = d->lengths ? resblock2_big_kernel<true> : resblock2_big_kernel<false>;
  static PerDeviceOnce configured[2];
  if (configured[d->lengths ? 1 : 0].first_use()) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  }
  const int resident_pairs = num_sms() / 2;
  const int pairs = p.n_pairs < resident_pairs ? p.n_pairs : resident_pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * pairs));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  count_launch();
  return 0;
}

}  // namespace avc
