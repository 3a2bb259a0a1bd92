// A whole stack of small-batch LSTM layers as ONE wavefront (see include/avc_b200.h: avc_lstm_stack_ws).
//
// avc_lstm_seq_ws runs one layer: a frame is a chain of L2 round trips (grid barrier, h slice, reduction) of about
// 4.3 us whatever the batch is, and the layers of a stack run one after another -- LstmDV (factory/LstmDV.py:12,20:
// 3 x LSTM(768), 1000 frames) spends 3 x 1000 such frames.  Layer l at frame t needs only layer l-1 at frame t and its own
// frame t-1, so the layers can run a fixed number of TICKS APART, all at once, on disjoint SMs, and the stack costs
// T + 2 (L - 1) ticks instead of L x T frames.
//
// For that the input projection of the layers above the first has to move into the recurrence (a dense projection in
// front needs the whole sequence of the layer below), and every weight has to stay on chip for the whole sequence:
//   layer 0:   z = xproj_0[t] (dense GEMM in front, as before)     + W_hh0 h0_{t-1}
//   layer l>0: z = bias_l + W_ih_l h^{l-1}_t                       + W_hh_l h^l_{t-1}
// The grid is L layers x R = 4H/128 row blocks x 2 CTAs, each pair a thread-block cluster; CTA s of a pair holds the K
// half s of its row block of W_hh and (above the first layer) of W_ih, ONE fp16 term each -- that is what fits: 128 rows
// x 768 channels x 2 bytes = 384 of the 512 tensor-memory columns per CTA beside two accumulators, 144 CTAs for LstmDV.
// (Two terms for every matrix would need 47 MB on chip.  One term costs precision: embedding rel-L2 2.7 .. 3.0e-4 instead
// of 1.5 .. 1.7e-4 on the test weights, 6.7e-4 instead of 3.5e-4 on the x3-gain stress weights, gate 1e-3 --
// scripts/lstm_stack_precision.py; the caller chooses.)
// The weights are the A operand of tcgen05.mma read from tensor memory.  Measured (profiles/r02_lstm_stack_v1_*): such an
// MMA takes ~85 cycles whatever its width, so the MMAs are the longest link of a tick's serial chain, and only those on
// h^l_{t-1} have to be on it: layer l runs TWO ticks behind layer l-1, so h^{l-1}_{t+1} already exists while frame t is
// being finished, and its product with W_ih is issued right behind the frame's own MMAs into the OTHER of two
// accumulators -- it runs while the cell warps, the reduction and the grid barrier of frame t are in flight.  At the
// next tick the W_hh products accumulate on top of it.  Per tick a CTA TMA-loads its K half of h^l_{t-1} (two groups, so
// the MMAs start on the first) and of h^{l-1}_{t+1}, issues H/32 + H/32 MMAs of width N = B', and the pair reduces its two
// partial sums through distributed shared memory exactly like avc_lstm_seq_ws (st.async crediting the owner's
// mbarrier); each CTA finalises 16 hidden units: cell update with c in registers, h_t written as fp16 into the stack's
// scratch sequence hs[l][t+1] (frame 0 is the zero initial state).  One release/acquire grid barrier per tick orders
// the h stores of tick k before the TMA reads of tick k + 1.
//
// Warp roles: 0 = grid barrier + operand producer, 1 = MMA issuer, 2..5 (2..9 at 64 utterances) = reduction + cell
// (warps 2, 3 store h_t).
#include <cuda_fp16.h>
#include <cstring>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

constexpr int kStMaxLayers = AVC_STACK_MAX_LAYERS;
constexpr int kStRowsOwn = kBlockM / 2;        // gate rows each CTA of the pair finalises
constexpr int kStUnitsOwn = kStRowsOwn / 4;    // = 16 hidden units
constexpr int kStGroups = 2;                   // load groups of the h^l_{t-1} operand (one mbarrier each)
constexpr int kStSkew = 2;                     // ticks between consecutive layers

struct alignas(64) StackParams {
  // hs[l] as (64 channels, B rows, H/64 chunks, T + 1 frames): one TMA operation brings a whole group of 64-channel
  // operand tiles (rows >= B and chunks >= H/64 are zero-filled)
  CUtensorMap tmap_c[kStMaxLayers];   // box {64, AR, ceil(H/128 / 2), 1}: a group of the K half of h^l_{t-1}
  CUtensorMap tmap_p[kStMaxLayers];   // box {64, AR, H/128, 1}: the K half of h^{l-1}_{t+1} (read by layer l + 1)
  const __half* w_ih[kStMaxLayers];   // l >= 1: [4H][H]
  const __half* w_hh[kStMaxLayers];   // [4H][H]
  const float* bias[kStMaxLayers];    // l >= 1: [4H]
  const float* xproj0;
  __half* hs;
  float* h_last;
  unsigned int* grid_barrier;
  long long* debug_clk;               // optional: 16 clock64 stamps per (tick, CTA)
  int B, T, H, L;
  const int* lengths;                 // optional [B]: h_last[n] is the top layer's h at frame lengths[n] - 1 (NULL: T - 1)
};

__device__ __forceinline__ uint32_t st_map_to_cta(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_f4(uint32_t addr, uint32_t mbar, float a, float b, float c, float d) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr),
               "f"(a), "f"(b), "f"(c), "f"(d), "r"(mbar)
               : "memory");
}

template <int AR>
struct StackCfg {
  // 64 utterances: two cell warps per TMEM lane quarter (each drains half of the accumulator columns and finalises half
  // of the cells) -- measured 1.0 K cycles per tick less than four warps walking everything twice
  static constexpr int kCellWarps = AR > 32 ? 8 : 4;
  static constexpr int kCellThreads = 32 * kCellWarps;
  static constexpr int kThreads = 64 + kCellThreads;
  static constexpr int NQ = AR / 4;                                   // groups of 4 utterances
  static constexpr int kItems = kStUnitsOwn * NQ;                     // (unit, utterance group) pairs an owner finalises
  static constexpr int IT = (kItems + kCellThreads - 1) / kCellThreads;
  static constexpr int kHTile = AR * kRowBytes;                       // one 64-channel chunk of the operand rows
  static constexpr int kRedFrameBytes = 2 * AR * kStRowsOwn * 4;      // what one tick pushes into an owner
  static constexpr int kRedBytes = (kRedFrameBytes + 1023) / 1024 * 1024;
  static constexpr int kStageBytes = (AR * kStUnitsOwn * 4 + 1023) / 1024 * 1024;
  static constexpr uint32_t kAccCols = AR < 32 ? 32 : AR;             // one accumulator; there are two
  // operand tiles: the h^l_{t-1} half in whole load groups (a zero-filled / unused tile when H/128 is odd), then the
  // h^{l-1}_{t+1} half
  __host__ __device__ static int crit_tiles(int H) { return kStGroups * ((H / 128 + kStGroups - 1) / kStGroups); }
  __host__ __device__ static int h_tiles(int H) { return crit_tiles(H) + H / 128; }
  static int smem_bytes(int H) { return h_tiles(H) * kHTile + kRedBytes + kStageBytes + 128 + 1024 /* alignment slack */; }
};

// RAGGED: h_last[n] at frame lengths[n] - 1.  A separate instantiation, because the per-utterance comparison changes
// the register allocation of the kernel; the fixed-length instantiation is the kernel as it is without lengths.
template <int AR, bool RAGGED>
__global__ void __launch_bounds__(StackCfg<AR>::kThreads, 1) lstm_stack_kernel(const __grid_constant__ StackParams p) {
  using Cfg = StackCfg<AR>;
  constexpr int NQ = Cfg::NQ, IT = Cfg::IT;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_h = base;
  float* s_red = reinterpret_cast<float*>(s_h + Cfg::h_tiles(p.H) * Cfg::kHTile);
  float* s_stage = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s_red) + Cfg::kRedBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_stage) + Cfg::kStageBytes);
  uint64_t* w_full = bars + 0;
  uint64_t* d_full = bars + 1;        // the frame's MMAs have completed (accumulator ready)
  uint64_t* red_full = bars + 2;      // both partial sums of the rows this CTA owns have landed
  uint64_t* epi_done = bars + 3;      // this CTA's h_t is stored (and the accumulator drained)
  uint64_t* h_full = bars + 4;        // [kStGroups]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int R = 4 * p.H / kBlockM;
  const int cid = blockIdx.x >> 1;
  const int layer = cid / R;
  const int r = cid % R;
  const unsigned int n_ctas = gridDim.x;
  long long* const clk = p.debug_clk;
#define AVC_ST_STAMP(k_, i_) \
  if (clk) clk[((long long)(k_) * n_ctas + blockIdx.x) * 16 + (i_)] = clock64()

  // this CTA multiplies the K half [k0, k0 + H/2) of W_hh (and of W_ih above the first layer): nc 64-channel chunks each
  const int nc = p.H / 128;
  const int k0c = (int)rank * nc;                                // first chunk of the half
  const int cpg = (nc + kStGroups - 1) / kStGroups;              // chunks per load group of the h^l_{t-1} operand
  const int ngroups = (nc + cpg - 1) / cpg;
  const bool upper = layer > 0;
  uint8_t* const s_hp = s_h + Cfg::crit_tiles(p.H) * Cfg::kHTile;   // tiles of h^{l-1}_{t+1}
  uint64_t* const h_pre = bars + 6;     // the K half of h^{l-1}_{t+1} has landed
  uint64_t* const pre_done = bars + 7;  // the MMAs that read it have completed (its tiles may be overwritten)

  if (threadIdx.x == 0) {
    mbar_init(w_full, Cfg::kCellWarps);
    mbar_init(d_full, 1);
    mbar_init(red_full, 1);
    mbar_init(epi_done, AR > 32 ? 2 : 1);     // one arrival per warp that stores h_t
    for (int g = 0; g < kStGroups; ++g) mbar_init(h_full + g, 1);
    mbar_init(h_pre, 1);
    mbar_init(pre_done, 1);
    fence_mbar_init();
    prefetch_tmap(&p.tmap_c[layer]);
    if (upper) prefetch_tmap(&p.tmap_p[layer - 1]);
  }
  constexpr uint32_t tmem_cols = 512;
  if (warp == 1) {
    tmem_alloc(tmem_ptr, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  cluster_sync_all();                 // the peer credits bytes to this CTA's red_full: its init must be visible cluster-wide
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
  const uint32_t tmem_w = tmem_base + 2 * Cfg::kAccCols;    // W_hh half at columns [0, 32 nc), W_ih half behind it
  const int nticks = p.T + kStSkew * (p.L - 1);

  if (warp == 0) {
    if (lane == 0) {
      for (int k = 0; k < nticks; ++k) {
        const int t = k - kStSkew * layer;     // the frame this CTA finishes at tick k (t = -1: only the W_ih part of frame 0)
        if (k > 0) {
          // this CTA's part of the previous tick's h is stored, then every CTA's
          if (t - 1 >= 0 && t - 1 < p.T) mbar_wait(epi_done, (t - 1) & 1);
          grid_arrive_wait(p.grid_barrier, (unsigned)k * n_ctas,
                           clk ? clk + ((long long)k * n_ctas + blockIdx.x) * 16 : nullptr);  // stamp 0: arrival issued
        }
        AVC_ST_STAMP(k, 1);
        const bool crit = t >= 0 && t < p.T, pre = upper && t + 1 >= 0 && t + 1 < p.T;
        if (crit || pre) fence_proxy_async_global();   // the operand rows were written with generic stores
        if (crit)
          for (int g = 0; g < ngroups; ++g) {
            mbar_arrive_expect_tx(h_full + g, cpg * Cfg::kHTile);          // the whole box, zero-filled part included
            tma_load_4d(s_h + g * cpg * Cfg::kHTile, &p.tmap_c[layer], h_full + g, 0, 0, k0c + g * cpg, t);
          }
        if (pre) {
          // h^{l-1}_{t+1} = frame t + 2 of the sequence below (stored a tick ago); its tiles are free once the MMAs of the
          // previous W_ih part have completed (long ago: they were issued a tick earlier)
          if (t + 1 > 0) mbar_wait(pre_done, t & 1);
          mbar_arrive_expect_tx(h_pre, nc * Cfg::kHTile);
          tma_load_4d(s_hp, &p.tmap_p[layer - 1], h_pre, 0, 0, k0c, t + 2);
        }
        if (clk && crit)                 // profiling only: when each group really landed (the MMA thread sees a group
          for (int g = 0; g < ngroups; ++g) {   // only after it has issued the previous group's MMAs)
            mbar_wait(h_full + g, t & 1);
            AVC_ST_STAMP(k, 11 + g);
          }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(kBlockM, AR, false) ^ kIdescF16Xor;
      mbar_wait(w_full, 0);
      tc_fence_after();
      for (int t = upper ? -1 : 0; t < p.T; ++t) {
        const int k = t + kStSkew * layer;
        if (t >= 0) {
          // frame t: W_hh h_{t-1} on top of the W_ih part issued a tick ago (layer 0: a fresh accumulator)
          const uint32_t acc = tmem_base + (t & 1) * Cfg::kAccCols;
          for (int g = 0; g < ngroups; ++g) {
            mbar_wait(h_full + g, t & 1);
            AVC_ST_STAMP(k, g == 0 ? 2 : 7 + g);                      // 2, 8: operand group g landed
            tc_fence_after();
            const int c0 = g * cpg, c1 = min(nc, c0 + cpg);
            for (int c = c0; c < c1; ++c) {
              const uint32_t h = smem_u32(s_h + c * Cfg::kHTile);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_bf16_ts(acc, tmem_w + c * 32 + kk * 8, umma_desc_sw128(h + kk * 32), idesc,
                             (!upper && c == 0 && kk == 0) ? 0u : 1u);
            }
          }
          umma_commit(d_full);
          AVC_ST_STAMP(k, 10);                                        // the frame's MMAs issued
        }
        if (upper && t + 1 < p.T) {
          // W_ih h^{l-1}_{t+1} into the other accumulator (drained two frames ago: that drain is ordered before these
          // MMAs through epi_done -> grid barrier -> h_pre), off the serial chain of the tick
          const uint32_t acc = tmem_base + ((t + 1) & 1) * Cfg::kAccCols;
          mbar_wait(h_pre, (t + 1) & 1);
          tc_fence_after();
          for (int c = 0; c < nc; ++c) {
            const uint32_t h = smem_u32(s_hp + c * Cfg::kHTile);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16_ts(acc, tmem_w + (nc + c) * 32 + kk * 8, umma_desc_sw128(h + kk * 32), idesc,
                           (c == 0 && kk == 0) ? 0u : 1u);
          }
          umma_commit(pre_done);
          AVC_ST_STAMP(k, 9);                                         // the W_ih part of the next frame issued
        }
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3;                           // TMEM lane quarter
    const int row = q * 32 + lane;                    // accumulator row = packed gate row within the row block
    const int ctid = threadIdx.x - 64;                // 0 .. kCellThreads - 1
    constexpr int HW = Cfg::kCellWarps / 4;           // warps per lane quarter
    const int half = (warp - 2) / 4;                  // which of them
    // reduction buffer of an owner: [source rank][group of 4 utterances][gate][owned unit][4] fp32 -- a warp's 16-byte
    // stores of one group fill one contiguous 512-byte run, and the cell threads of adjacent units read adjacent float4
    const uint32_t owner = row / kStRowsOwn;
    const int slot = (row & 3) * kStUnitsOwn + (row % kStRowsOwn) / 4;
    const uint32_t push_addr = st_map_to_cta(smem_u32(s_red + ((int)rank * NQ * kStRowsOwn + slot) * 4), owner);
    const uint32_t owner_bar = st_map_to_cta(smem_u32(red_full), owner);
    // the half of the rows this CTA owns itself stays local (plain shared-memory stores + a barrier among the cell warps):
    // only the peer's half crosses the cluster (~21 B/clk: 16 KB per tick at 64 utterances)
    const bool local = owner == rank;
    float* const local_ptr = s_red + ((int)rank * NQ * kStRowsOwn + slot) * 4;
    {
      // this thread's W rows -> its TMEM lane, once: 32 fp16 (16 columns) per store; W_hh half, then W_ih half
      const uint32_t lane_base = tmem_w + (static_cast<uint32_t>(q * 32) << 16);
      for (int m = 0; m < (upper ? 2 : 1); ++m) {
        const __half* w = m == 0 ? p.w_hh[layer] : p.w_ih[layer];
        const uint4* srcw = reinterpret_cast<const uint4*>(w + ((long long)r * kBlockM + row) * p.H + k0c * 64);
        for (int g = half * (2 * nc / HW); g < (half + 1) * (2 * nc / HW); ++g) {
          uint32_t v[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 u = __ldg(srcw + g * 4 + i);
            v[4 * i] = u.x; v[4 * i + 1] = u.y; v[4 * i + 2] = u.z; v[4 * i + 3] = u.w;
          }
          tmem_st_32x16(lane_base + m * nc * 32 + g * 16, v);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(w_full);
    }
    int u_own[IT], n4[IT];
    bool active[IT];
    float4 bias4[IT];
    float c_state[IT][4];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      const int e = it * Cfg::kCellThreads + ctid;    // adjacent threads: adjacent units (contiguous reads)
      u_own[it] = e % kStUnitsOwn;
      n4[it] = e / kStUnitsOwn;
      active[it] = n4[it] < NQ;
      bias4[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (layer > 0)
        bias4[it] = __ldg(reinterpret_cast<const float4*>(p.bias[layer] + r * kBlockM +
                                                          4 * ((int)rank * kStUnitsOwn + u_own[it])));
#pragma unroll
      for (int j = 0; j < 4; ++j) c_state[it][j] = 0.f;
    }
    const long long H4 = 4LL * p.H;
    __half* const hs_l = p.hs + (long long)layer * (p.T + 1) * p.B * p.H;
    const bool top = layer == p.L - 1;
    for (int t = 0; t < p.T; ++t) {
      // the additive term of this thread's cells: issued first, consumed after the reduction
      float z[IT][4][4];                              // [item][utterance j][gate]
#pragma unroll
      for (int it = 0; it < IT; ++it)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 xp = bias4[it];
          const int n = n4[it] * 4 + j;
          if (layer == 0 && active[it] && n < p.B)
            xp = __ldg(reinterpret_cast<const float4*>(p.xproj0 + ((long long)n * p.T + t) * H4 + r * kBlockM +
                                                       4 * ((int)rank * kStUnitsOwn + u_own[it])));
          z[it][j][0] = xp.x; z[it][j][1] = xp.y; z[it][j][2] = xp.z; z[it][j][3] = xp.w;
        }
      if (threadIdx.x == 64) mbar_arrive_expect_tx(red_full, Cfg::kRedFrameBytes / 2);   // the peer's half
      mbar_wait(d_full, t & 1);
      if (threadIdx.x == 64) AVC_ST_STAMP(t + kStSkew * layer, 3);
      tc_fence_after();
      // this thread's accumulator row, pushed to the CTA that owns it
      {
        constexpr int JN = AR / 16 / HW;              // groups of 16 utterances this warp drains
        uint32_t a[JN][16];
#pragma unroll
        for (int jj = 0; jj < JN; ++jj)
          tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (t & 1) * Cfg::kAccCols + (half * JN + jj) * 16,
                        a[jj]);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < JN; ++jj)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int grp = (half * JN + jj) * 4 + i;             // group of 4 utterances
            if (local)
              *reinterpret_cast<float4*>(local_ptr + grp * kStRowsOwn * 4) =
                  make_float4(__uint_as_float(a[jj][i * 4]), __uint_as_float(a[jj][i * 4 + 1]),
                              __uint_as_float(a[jj][i * 4 + 2]), __uint_as_float(a[jj][i * 4 + 3]));
            else
              st_async_f4(push_addr + grp * kStRowsOwn * 16, owner_bar, __uint_as_float(a[jj][i * 4]),
                          __uint_as_float(a[jj][i * 4 + 1]), __uint_as_float(a[jj][i * 4 + 2]),
                          __uint_as_float(a[jj][i * 4 + 3]));
          }
      }
      tc_fence_before();                // accumulator reads before the next frame's MMAs (via epi_done -> h_full)
      if (threadIdx.x == 64) AVC_ST_STAMP(t + kStSkew * layer, 4);
      asm volatile("bar.sync 2, %0;" ::"n"(Cfg::kCellThreads) : "memory");   // the local half is in place
      mbar_wait_cluster(red_full, t & 1);
      if (threadIdx.x == 64) AVC_ST_STAMP(t + kStSkew * layer, 5);
#pragma unroll
      for (int it = 0; it < IT; ++it) {
        if (!active[it]) continue;
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float4 v = *reinterpret_cast<const float4*>(
                s_red + ((s * NQ + n4[it]) * kStRowsOwn + g * kStUnitsOwn + u_own[it]) * 4);   // gate g, 4 utterances
            z[it][0][g] += v.x; z[it][1][g] += v.y; z[it][2][g] += v.z; z[it][3][g] += v.w;
          }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float cn, hn;
          lstm_cell(z[it][j][0], z[it][j][1], z[it][j][2], z[it][j][3], c_state[it][j], cn, hn);
          c_state[it][j] = cn;
          s_stage[(n4[it] * 4 + j) * kStUnitsOwn + u_own[it]] = hn;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kCellThreads) : "memory");
      if (threadIdx.x == 64) AVC_ST_STAMP(t + kStSkew * layer, 6);
      if (warp == 2 || (AR > 32 && warp == 3)) {
        // utterance n: the 16 units this CTA finalised = 32 bytes of fp16 in frame t + 1 of this layer's sequence
        const int n = (warp - 2) * 32 + lane;
        if (n < AR && n < p.B) {
          const int ug = r * 32 + (int)rank * kStUnitsOwn;
          const float4* sv = reinterpret_cast<const float4*>(s_stage + n * kStUnitsOwn);
          const float4 h0 = sv[0], h1 = sv[1], h2 = sv[2], h3 = sv[3];
          uint4* o = reinterpret_cast<uint4*>(hs_l + ((long long)(t + 1) * p.B + n) * p.H + ug);
          o[0] = make_uint4(pack_f16(h0.x, h0.y), pack_f16(h0.z, h0.w), pack_f16(h1.x, h1.y), pack_f16(h1.z, h1.w));
          o[1] = make_uint4(pack_f16(h2.x, h2.y), pack_f16(h2.z, h2.w), pack_f16(h3.x, h3.y), pack_f16(h3.z, h3.w));
          if (top && (RAGGED ? is_last_frame(p.lengths, n, t, p.T) : t == p.T - 1) && p.h_last) {
            float4* hl = reinterpret_cast<float4*>(p.h_last + (long long)n * p.H + ug);
            hl[0] = h0; hl[1] = h1; hl[2] = h2; hl[3] = h3;
          }
          fence_proxy_async_global();   // order the h stores before later async-proxy (TMA) reads
        }
        __syncwarp();
        if (lane == 0) {
          AVC_ST_STAMP(t + kStSkew * layer, 7);
          mbar_arrive(epi_done);        // after bar.sync 1: every cell warp has drained the accumulator too
        }
      }
    }
  }
#undef AVC_ST_STAMP
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();                   // no CTA may exit while its peer can still push into its shared memory
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

template <int AR, bool RAGGED>
static int launch_stack(const StackParams& p, const avc_lstm_stack_desc* d, cudaStream_t stream) {
  using Cfg = StackCfg<AR>;
  auto kern = lstm_stack_kernel<AR, RAGGED>;
  const int smem = Cfg::smem_bytes(d->H);
  AVC_REQUIRE(smem <= 227 * 1024, "avc_lstm_stack_ws: H=%d B=%d needs %d bytes of shared memory", d->H, d->B, smem);
  static int configured[PerDeviceOnce::kMaxDevices] = {};   // largest size set so far, per device
  int dev = 0;
  AVC_CHECK_CUDA(cudaGetDevice(&dev));
  const bool known = dev >= 0 && dev < PerDeviceOnce::kMaxDevices;
  if (!known || configured[dev] < smem) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (known) configured[dev] = smem;
  }
  const int grid = d->L * (4 * d->H / kBlockM) * 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(Cfg::kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  const int rc = persistent_launch_config(cfg, attr, reinterpret_cast<const void*>(kern), 2, "avc_lstm_stack_ws");
  if (rc != 0) return rc;
  AVC_CHECK_CUDA(cudaMemsetAsync(d->grid_barrier, 0, sizeof(unsigned int), stream));
  // frame 0 of every layer's sequence: the zero initial state
  const size_t frame_bytes = (size_t)d->B * d->H * 2, layer_bytes = frame_bytes * (size_t)(d->T + 1);
  for (int l = 0; l < d->L; ++l)
    AVC_CHECK_CUDA(cudaMemsetAsync(static_cast<uint8_t*>(d->hs) + l * layer_bytes, 0, frame_bytes, stream));
  AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  count_launch();
  return 0;
}

}  // namespace avc

extern "C" int avc_lstm_stack_ws(const avc_lstm_stack_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_lstm_stack_ws: null descriptor");
  AVC_REQUIRE(d->B > 0 && d->B <= 64 && d->T > 0, "avc_lstm_stack_ws: B=%d T=%d (1 <= B <= 64)", d->B, d->T);
  AVC_REQUIRE(d->L >= 1 && d->L <= kStMaxLayers, "avc_lstm_stack_ws: L=%d (1..%d layers)", d->L, kStMaxLayers);
  AVC_REQUIRE(d->H > 0 && d->H % 128 == 0 && d->H / 2 + 128 <= 512,
              "avc_lstm_stack_ws: unsupported H=%d (multiple of 128, at most 768: the weights of a CTA fill H/2 "
              "tensor-memory columns beside the two accumulators)", d->H);
  AVC_REQUIRE(d->xproj0 && d->w_hh[0] && d->hs && d->grid_barrier, "avc_lstm_stack_ws: missing buffer");
  for (int l = 1; l < d->L; ++l)
    AVC_REQUIRE(d->w_ih[l] && d->w_hh[l] && d->bias[l], "avc_lstm_stack_ws: missing weights of layer %d", l);
  if (d->L * (4 * d->H / kBlockM) * 2 > num_sms()) {
    set_error("avc_lstm_stack_ws: %d layers x %d row blocks x 2 CTAs exceed the %d SMs", d->L, 4 * d->H / kBlockM, num_sms());
    return AVC_ERR_NOT_RESIDENT;
  }
  const uint64_t H = (uint64_t)d->H;
  const int ar = d->B <= 16 ? 16 : (d->B <= 32 ? 32 : 64);
  StackParams p;
  memset(&p, 0, sizeof(p));
  const uint64_t frame_bytes = (uint64_t)d->B * H * 2, layer_bytes = frame_bytes * (uint64_t)(d->T + 1);
  const uint32_t nc = (uint32_t)(d->H / 128);
  const uint64_t dh[4] = {64, (uint64_t)d->B, H / 64, (uint64_t)d->T + 1};
  const uint64_t sh[3] = {H * 2, 128, frame_bytes};
  const uint32_t box_c[4] = {64, (uint32_t)ar, (nc + kStGroups - 1) / kStGroups, 1}, box_p[4] = {64, (uint32_t)ar, nc, 1};
  for (int l = 0; l < d->L; ++l) {
    const void* seq = static_cast<uint8_t*>(d->hs) + l * layer_bytes;
    if (!encode_tmap_4d(&p.tmap_c[l], 2, seq, dh, sh, box_c) || !encode_tmap_4d(&p.tmap_p[l], 2, seq, dh, sh, box_p)) return -3;
    p.w_ih[l] = static_cast<const __half*>(d->w_ih[l]);
    p.w_hh[l] = static_cast<const __half*>(d->w_hh[l]);
    p.bias[l] = d->bias[l];
  }
  p.xproj0 = d->xproj0;
  p.hs = static_cast<__half*>(d->hs);
  p.h_last = d->h_last;
  p.lengths = d->lengths;
  p.grid_barrier = d->grid_barrier;
  p.debug_clk = d->debug_clk;
  p.B = d->B;
  p.T = d->T;
  p.H = d->H;
  p.L = d->L;
  if (p.lengths)
    return ar == 16 ? launch_stack<16, true>(p, d, stream) : ar == 32 ? launch_stack<32, true>(p, d, stream)
                                                          : launch_stack<64, true>(p, d, stream);
  return ar == 16 ? launch_stack<16, false>(p, d, stream) : ar == 32 ? launch_stack<32, false>(p, d, stream)
                                                         : launch_stack<64, false>(p, d, stream);
}
