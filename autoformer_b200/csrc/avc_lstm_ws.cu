// Small-batch LSTM recurrence with the recurrent weights STATIONARY on chip (see include/avc_b200.h:
// avc_lstm_seq_ws).  B <= 64 utterances, split-bf16 or fp16x2 precision.
//
// At a small batch the batched kernel (avc_lstm.cu) multiplies a 128-row activation tile of which only B rows are real
// and re-streams every weight tile from L2 each frame; a frame costs ~15 K cycles whatever B is.  Here the roles of the
// operands are swapped:
//   z^T [4H x B] = W_hh [4H x H] . h_{t-1}^T [H x B]
// W is the M-side operand and never moves: the grid is R = 4H / 128 row blocks x S K-slices, and CTA (r, s) keeps
// W[128 r .. 128 r + 128, slice s] (hi and lo halves, <= 128 KB) on chip for the whole sequence -- in tensor memory, as
// the A operand of tcgen05.mma.  Per frame a
// CTA loads only its K-slice of h_{t-1} (B rows: a few KB), issues
//   W_hi x [h_hi ; h_lo]   (one MMA of width N = 2 B')      and      W_lo x h_hi   (N = B')
// into a 128 x 2B' accumulator, and the S CTAs of a row block -- one thread-block CLUSTER -- reduce their partial sums
// through distributed shared memory: every accumulator row is pushed to the CTA that owns it with st.async, which
// credits the bytes to the owner's mbarrier (no fence, no separate arrival).  Gate rows are packed
// p = 128 (u / 32) + 4 (u % 32) + gate, so the 128 / S rows an owner finalises are whole hidden units: it adds xproj,
// runs the cell (c stays in registers for all T frames) and writes h_t in the split operand format.
// The frame ends with the same release/acquire grid barrier as the batched kernel (every CTA needs all of h_t).
// Two barrier-free variants were built and measured slower (B = 32, H = 1024, cycles per frame; barrier: 8.1 K):
//  - per-CTA progress flags, each consumer polling only the H / 32 CTAs that produce its K-slice: 10.9 K;
//  - h_t exchanged in a flag-carrying format (8-byte words {2 bf16, frame tag}, no fence, no counter, consumers poll
//    the data itself): 26.7 K at B = 32 (every CTA re-reads 64 KB of tagged words per poll round), 7.4 K at B = 1
//    against 7.2 K with the barrier.
// Without the barrier the CTAs of a cluster drift up to one frame apart and the time comes back as waiting in the
// reduction and before the MMAs; the slowest of the producers sets the pace either way.
//
// Warp roles: 0 = grid barrier + h_{t-1} producer, 1 = MMA issuer, 2..5 = reduction + cell (warp 2 stores h_t).
#include <cuda_bf16.h>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

constexpr int kWsThreads = 192;
constexpr int kWsCellWarps = 4;

struct alignas(64) WsParams {
  const __nv_bfloat16* w; // w_hh [4H][2H]
  CUtensorMap tmap_h;     // hseq as (H, B, part, T), box {64, AR, 2, 1}
  const float* xproj;
  __nv_bfloat16* hseq;
  float* hseq_f32;
  float* h_last;
  unsigned int* grid_barrier;
  long long* debug_clk;   // optional: 8 clock64 stamps per (frame, CTA)
  int B, T, H;
  int chunks;             // 64-channel chunks of this CTA's K-slice
  const int* lengths;     // optional [B]: h_last[n] is h at frame lengths[n] - 1 (NULL: T - 1)
};

template <int AR, int S>
struct WsCfg {
  static constexpr int kRowsOwn = kBlockM / S;        // gate rows each CTA of the cluster finalises
  static constexpr int kUnitsOwn = kRowsOwn / 4;
  // reduction buffer of an owner: [source rank s][utterance n][owned row] fp32 -- for one utterance the rows of a
  // warp are consecutive, so every remote store instruction of the push is one contiguous 128-byte segment
  static constexpr int kHTile = AR * kRowBytes;       // one part of one chunk
  static constexpr int kRedFrameBytes = S * AR * kRowsOwn * 4;       // what one frame pushes into an owner
  static constexpr int kRedBytes = (kRedFrameBytes + 1023) / 1024 * 1024;
  static constexpr int kStageBytes = (AR * kUnitsOwn * 4 + 1023) / 1024 * 1024;
  static constexpr uint32_t kAccCols = 2 * AR < 32 ? 32 : 2 * AR;
  // tensor memory: the accumulator, then this CTA's W slice as the A operand: [hi: 32 chunks columns | lo]
  __host__ __device__ static uint32_t tmem_cols(int chunks) {
    uint32_t need = kAccCols + 64u * chunks, c = 32;
    while (c < need) c *= 2;
    return c;
  }
  static int smem_bytes(int chunks, bool f16) {
    return chunks * (f16 ? 1 : 2) * kHTile + kRedBytes + kStageBytes + 128 + 1024 /* alignment slack */;
  }
};

__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// 16-byte store into a cluster peer's shared memory that credits its bytes to the peer's mbarrier on completion
__device__ __forceinline__ void st_async_f4(uint32_t addr, uint32_t mbar, float4 v) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(mbar)
               : "memory");
}
// (mbar_wait_cluster: the cluster-scope acquire wait lives in avc_ptx.cuh)

// F16 ("fp16x2" precision): h is one fp16 value per unit, the weights two fp16 terms; both products W_hi x h and
// W_lo x h are N = AR MMAs onto the SAME accumulator columns.
template <int AR, int S, bool F16>
__global__ void __launch_bounds__(kWsThreads, 1) lstm_ws_kernel(const __grid_constant__ WsParams p) {
  using Cfg = WsCfg<AR, S>;
  constexpr int HP = F16 ? 1 : 2;                    // tiles of h per 64-channel chunk (hi / lo halves)
  constexpr int NQ = AR / 4;                         // groups of 4 utterances
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_h = base;
  float* s_red = reinterpret_cast<float*>(s_h + p.chunks * HP * Cfg::kHTile);
  float* s_stage = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s_red) + Cfg::kRedBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_stage) + Cfg::kStageBytes);
  uint64_t* w_full = bars + 0;
  uint64_t* d_full = bars + 1;        // the frame's MMAs have completed (accumulator ready)
  uint64_t* red_full = bars + 2;      // all partial sums of the rows this CTA owns have landed
  uint64_t* epi_done = bars + 3;      // this CTA's h_t is stored (and the accumulator drained)
  uint64_t* h_full = bars + 4;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();           // K-slice
  const int r = blockIdx.x / S;                      // row block
  const int k0 = (int)rank * p.chunks * 64;
  const unsigned int n_ctas = gridDim.x;
  long long* const clk = p.debug_clk;
#define AVC_WS_STAMP(t_, i_) \
  if (clk) clk[((long long)(t_) * n_ctas + blockIdx.x) * 8 + (i_)] = clock64()

  if (threadIdx.x == 0) {
    mbar_init(w_full, kWsCellWarps);
    mbar_init(h_full, 1);
    mbar_init(d_full, 1);
    mbar_init(red_full, 1);
    mbar_init(epi_done, AR > 32 ? 2 : 1);     // one arrival per warp that stores h_t
    fence_mbar_init();
    prefetch_tmap(&p.tmap_h);
  }
  const uint32_t tmem_cols = Cfg::tmem_cols(p.chunks);
  if (warp == 1) {
    tmem_alloc(tmem_ptr, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  cluster_sync_all();                 // peers credit bytes to this CTA's red_full: its init must be visible cluster-wide
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
  const uint32_t tmem_w = tmem_base + Cfg::kAccCols;        // W_hi at columns [0, 32 chunks), W_lo behind it

  if (warp == 0) {
    if (lane == 0) {
      for (int t = 1; t < p.T; ++t) {
        // h_{t-1}: this CTA's part is stored, then every CTA's
        mbar_wait(epi_done, (t - 1) & 1);
        grid_arrive_wait(p.grid_barrier, (unsigned)t * n_ctas,
                         clk ? clk + ((long long)t * n_ctas + blockIdx.x) * 8 : nullptr);   // stamp 0: arrival issued
        AVC_WS_STAMP(t, 1);
        fence_proxy_async_global();     // h_{t-1} was written with generic stores
        // (one mbarrier per chunk, so that the MMAs start on the first chunk, measured slower: +430 cycles per frame)
        mbar_arrive_expect_tx(h_full, p.chunks * HP * Cfg::kHTile);
        for (int c = 0; c < p.chunks; ++c)
          tma_load_4d(s_h + c * HP * Cfg::kHTile, &p.tmap_h, h_full, k0 + c * 64, 0, 0, t - 1);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t wide = umma_idesc(kBlockM, 2 * AR, false), narrow = umma_idesc(kBlockM, AR, false);
      mbar_wait(w_full, 0);
      tc_fence_after();
      for (int t = 1; t < p.T; ++t) {
        // (the accumulator is free: h_{t-1} exists only after this CTA's cell warps drained frame t - 1)
        mbar_wait(h_full, (t - 1) & 1);
        AVC_WS_STAMP(t, 2);
        tc_fence_after();               // orders the cell warps' accumulator reads of frame t - 1 before these MMAs
        for (int c = 0; c < p.chunks; ++c) {
          const uint32_t h = smem_u32(s_h + c * HP * Cfg::kHTile);           // [h_hi rows ; h_lo rows] (F16: h rows)
          if (F16) {
            const uint32_t w_hi = tmem_w + c * 32, w_lo = w_hi + p.chunks * 32;   // 8 columns per K = 16
            constexpr uint32_t idesc16 = umma_idesc(kBlockM, AR, false) ^ kIdescF16Xor;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(tmem_base, w_hi + k * 8, umma_desc_sw128(h + k * 32), idesc16, (c == 0 && k == 0) ? 0u : 1u);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(tmem_base, w_lo + k * 8, umma_desc_sw128(h + k * 32), idesc16, 1u);
          } else {
            const uint32_t w_hi = tmem_w + c * 32, w_lo = w_hi + p.chunks * 32;   // 8 columns per K = 16
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(tmem_base, w_hi + k * 8, umma_desc_sw128(h + k * 32), wide, (c == 0 && k == 0) ? 0u : 1u);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(tmem_base, w_lo + k * 8, umma_desc_sw128(h + k * 32), narrow, 1u);
          }
        }
        umma_commit(d_full);
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3;                           // TMEM lane quarter
    const int row = q * 32 + lane;                    // accumulator row = packed gate row within the row block
    const int e = (warp - 2) * 32 + lane;             // owner-phase index
    const int u_own = e % Cfg::kUnitsOwn, n4 = e / Cfg::kUnitsOwn;   // adjacent lanes: adjacent units (contiguous reads)
    const bool active = n4 < NQ;
    // reduction buffer of an owner: [source rank][group of 4 utterances][gate][owned unit][4] fp32 -- a warp's
    // 16-byte stores of one group fill one contiguous 512-byte run, and the cell threads of adjacent units read
    // adjacent float4 (no bank conflicts)
    const uint32_t owner = row / Cfg::kRowsOwn;
    const int slot = (row & 3) * Cfg::kUnitsOwn + (row % Cfg::kRowsOwn) / 4;
    const uint32_t push_addr = map_to_cta(smem_u32(s_red + ((int)rank * NQ * Cfg::kRowsOwn + slot) * 4), owner);
    const uint32_t owner_bar = map_to_cta(smem_u32(red_full), owner);
    // this thread's W row -> its TMEM lane, once: 32 bf16 (16 columns) per store, hi half then lo half
    const uint4* src = reinterpret_cast<const uint4*>(p.w + ((long long)r * kBlockM + row) * (2LL * p.H) + k0);
    const uint32_t lane_base = tmem_w + (static_cast<uint32_t>(q * 32) << 16);
    for (int part = 0; part < 2; ++part)
      for (int g = 0; g < 2 * p.chunks; ++g) {
        uint32_t v[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 u = __ldg(src + part * (p.H / 8) + g * 4 + i);
          v[4 * i] = u.x; v[4 * i + 1] = u.y; v[4 * i + 2] = u.z; v[4 * i + 3] = u.w;
        }
        tmem_st_32x16(lane_base + part * p.chunks * 32 + g * 16, v);
      }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(w_full);
    float c_state[4] = {0.f, 0.f, 0.f, 0.f};
    const long long H4 = 4LL * p.H;
    for (int t = 0; t < p.T; ++t) {
      // xproj of this thread's cells: issued first, consumed after the reduction
      float4 xp[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n4 * 4 + j;
        xp[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (active && n < p.B)
          xp[j] = __ldg(reinterpret_cast<const float4*>(p.xproj + ((long long)n * p.T + t) * H4 + r * kBlockM +
                                                        4 * ((int)rank * Cfg::kUnitsOwn + u_own)));
      }
      float z[4][4];                                  // [utterance j][gate]
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        z[j][0] = xp[j].x; z[j][1] = xp[j].y; z[j][2] = xp[j].z; z[j][3] = xp[j].w;
      }
      if (t > 0) {
        if (threadIdx.x == 64) mbar_arrive_expect_tx(red_full, Cfg::kRedFrameBytes);
        mbar_wait(d_full, (t - 1) & 1);
        if (threadIdx.x == 64) AVC_WS_STAMP(t, 3);
        tc_fence_after();
        // this thread's accumulator row: partial[n] = D[n] + D[AR + n]; pushed to the CTA that owns the row
#pragma unroll
        for (int j = 0; j < AR / 16; ++j) {
          uint32_t a[16], b[16];
          tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + j * 16, a);
          if (!F16) tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + AR + j * 16, b);
          tmem_ld_wait();
          if (F16) {
#pragma unroll
            for (int i = 0; i < 16; ++i) b[i] = 0u;       // +0.0f: one accumulator block only
          }
#pragma unroll
          for (int i = 0; i < 4; ++i)
            st_async_f4(push_addr + (j * 4 + i) * Cfg::kRowsOwn * 16, owner_bar,
                        make_float4(__uint_as_float(a[i * 4]) + __uint_as_float(b[i * 4]),
                                    __uint_as_float(a[i * 4 + 1]) + __uint_as_float(b[i * 4 + 1]),
                                    __uint_as_float(a[i * 4 + 2]) + __uint_as_float(b[i * 4 + 2]),
                                    __uint_as_float(a[i * 4 + 3]) + __uint_as_float(b[i * 4 + 3])));
        }
        tc_fence_before();              // accumulator reads before the next frame's MMAs (via epi_done -> h_full)
        if (threadIdx.x == 64) AVC_WS_STAMP(t, 4);
        mbar_wait_cluster(red_full, (t - 1) & 1);
        if (threadIdx.x == 64) AVC_WS_STAMP(t, 5);
        if (active) {
          const float* red = s_red;
#pragma unroll
          for (int s = 0; s < S; ++s)
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const float4 v = *reinterpret_cast<const float4*>(
                  red + ((s * NQ + n4) * Cfg::kRowsOwn + g * Cfg::kUnitsOwn + u_own) * 4);   // gate g, utterances 4 n4 .. + 3
              z[0][g] += v.x; z[1][g] += v.y; z[2][g] += v.z; z[3][g] += v.w;
            }
        }
      }
      if (active) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float cn, hn;
          lstm_cell(z[j][0], z[j][1], z[j][2], z[j][3], c_state[j], cn, hn);
          c_state[j] = cn;
          s_stage[(n4 * 4 + j) * Cfg::kUnitsOwn + u_own] = hn;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kWsCellWarps) : "memory");
      if (threadIdx.x == 64) AVC_WS_STAMP(t, 6);
      if (warp == 2 || (AR > 32 && warp == 3)) {
        // utterance n: the kUnitsOwn units this CTA finalised, as whole 8-byte groups of the split operand format
        // (one lane per utterance: warp 2 alone up to 32 utterances, warps 2 and 3 for 64)
        for (int n = (warp - 2) * 32 + lane; n < AR && n < p.B; n += AR) {
          const long long orow = (long long)n * p.T + t;
          const int ug = r * 32 + (int)rank * Cfg::kUnitsOwn;
#pragma unroll
          for (int i = 0; i < Cfg::kUnitsOwn / 4; ++i) {
            const float4 h = *reinterpret_cast<const float4*>(s_stage + n * Cfg::kUnitsOwn + i * 4);
            const float lx = h.x - __bfloat162float(__float2bfloat16_rn(h.x));
            const float ly = h.y - __bfloat162float(__float2bfloat16_rn(h.y));
            const float lz = h.z - __bfloat162float(__float2bfloat16_rn(h.z));
            const float lw = h.w - __bfloat162float(__float2bfloat16_rn(h.w));
            if (F16) {
              *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.hseq) + orow * p.H + ug + i * 4) =
                  make_uint2(pack_f16(h.x, h.y), pack_f16(h.z, h.w));
            } else {
              __nv_bfloat16* o = p.hseq + orow * (2LL * p.H) + ug + i * 4;
              *reinterpret_cast<uint2*>(o) = make_uint2(pack_bf16(h.x, h.y), pack_bf16(h.z, h.w));
              *reinterpret_cast<uint2*>(o + p.H) = make_uint2(pack_bf16(lx, ly), pack_bf16(lz, lw));
            }
            if (p.hseq_f32) *reinterpret_cast<float4*>(p.hseq_f32 + orow * p.H + ug + i * 4) = h;
            if (p.h_last && is_last_frame(p.lengths, n, t, p.T)) *reinterpret_cast<float4*>(p.h_last + (long long)n * p.H + ug + i * 4) = h;
          }
          fence_proxy_async_global();   // order the h stores before later async-proxy (TMA) reads
        }
        __syncwarp();
        if (lane == 0) {
          AVC_WS_STAMP(t, 7);
          mbar_arrive(epi_done);        // after bar.sync 1: every cell warp has drained the accumulator too
        }
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();                   // no CTA may exit while a peer can still push into its shared memory
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

template <int AR, int S, bool F16>
static int launch_ws(WsParams p, const avc_lstm_ws_desc* d, cudaStream_t stream) {
  using Cfg = WsCfg<AR, S>;
  auto kern = lstm_ws_kernel<AR, S, F16>;
  const int smem = Cfg::smem_bytes(p.chunks, F16);
  AVC_REQUIRE(smem <= 227 * 1024, "avc_lstm_seq_ws: H=%d B=%d needs %d bytes of shared memory", d->H, d->B, smem);
  static int configured[PerDeviceOnce::kMaxDevices] = {};   // largest size set so far, per device
  int dev = 0;
  AVC_CHECK_CUDA(cudaGetDevice(&dev));
  const bool known = dev >= 0 && dev < PerDeviceOnce::kMaxDevices;
  if (!known || configured[dev] < smem) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    if (known) configured[dev] = smem;
  }
  const int grid = 4 * d->H / kBlockM * S;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kWsThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  const int rc = persistent_launch_config(cfg, attr, reinterpret_cast<const void*>(kern), S, "avc_lstm_seq_ws");
  if (rc != 0) return rc;
  AVC_CHECK_CUDA(cudaMemsetAsync(d->grid_barrier, 0, sizeof(unsigned int), stream));
  AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  count_launch();
  return 0;
}

}  // namespace avc

extern "C" int avc_lstm_seq_ws(const avc_lstm_ws_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_lstm_seq_ws: null descriptor");
  AVC_REQUIRE(d->B > 0 && d->B <= 64 && d->T > 0, "avc_lstm_seq_ws: B=%d T=%d (1 <= B <= 64)", d->B, d->T);
  AVC_REQUIRE(d->xproj && d->w_hh && d->hseq && d->grid_barrier, "avc_lstm_seq_ws: missing buffer");
  AVC_REQUIRE(d->H > 0 && d->H % 256 == 0, "avc_lstm_seq_ws: unsupported H=%d (multiple of 256)", d->H);
  const uint64_t H = (uint64_t)d->H;
  const int ar = d->B <= 16 ? 16 : (d->B <= 32 ? 32 : 64);
  WsParams p;
  memset(&p, 0, sizeof(p));
  AVC_REQUIRE((reinterpret_cast<uintptr_t>(d->w_hh) & 15u) == 0, "avc_lstm_seq_ws: w_hh is not 16-byte aligned");
  AVC_REQUIRE(d->dtype == 0 || d->dtype == AVC_DTYPE_BF16X3 || d->dtype == AVC_DTYPE_F16, "avc_lstm_seq_ws: dtype %d",
              d->dtype);
  const bool f16 = d->dtype == AVC_DTYPE_F16;          // h: one fp16 per unit; else [hi | lo] bf16
  const uint64_t hp = f16 ? 1 : 2;
  const uint64_t dh[4] = {H, (uint64_t)d->B, hp, (uint64_t)d->T};
  const uint64_t sh[3] = {(uint64_t)d->T * hp * H * 2, H * 2, hp * H * 2};
  const uint32_t bh[4] = {64, (uint32_t)ar, (uint32_t)hp, 1};
  if (!encode_tmap_4d(&p.tmap_h, 2, d->hseq, dh, sh, bh)) return -3;
  p.w = static_cast<const __nv_bfloat16*>(d->w_hh);
  p.xproj = d->xproj;
  p.hseq = static_cast<__nv_bfloat16*>(d->hseq);
  p.hseq_f32 = d->hseq_f32;
  p.h_last = d->h_last;
  p.lengths = d->lengths;
  p.grid_barrier = d->grid_barrier;
  p.debug_clk = d->debug_clk;
  p.B = d->B;
  p.T = d->T;
  p.H = d->H;
  // K-slices per row block: 8 when the 4H/128 x 8 grid fits one wave as clusters of 8 (GPC granularity decides;
  // the occupancy query in launch_ws is the judge), else 4
  const int R = 4 * d->H / kBlockM;
#define AVC_WS_DISPATCH(S_)                                                                     \
  if (d->H % (64 * S_) == 0 && R * S_ <= num_sms()) {                                           \
    p.chunks = d->H / S_ / 64;                                                                  \
    const int rc = f16 ? (ar == 16   ? launch_ws<16, S_, true>(p, d, stream)                    \
                          : ar == 32 ? launch_ws<32, S_, true>(p, d, stream)                    \
                                     : launch_ws<64, S_, true>(p, d, stream))                   \
                       : (ar == 16   ? launch_ws<16, S_, false>(p, d, stream)                   \
                          : ar == 32 ? launch_ws<32, S_, false>(p, d, stream)                   \
                                     : launch_ws<64, S_, false>(p, d, stream));                 \
    if (rc != AVC_ERR_NOT_RESIDENT) return rc;                                                  \
  }
  AVC_WS_DISPATCH(8)
  AVC_WS_DISPATCH(4)
#undef AVC_WS_DISPATCH
  return AVC_ERR_NOT_RESIDENT;
}
