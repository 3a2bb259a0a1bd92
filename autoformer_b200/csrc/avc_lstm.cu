// Large-H LSTM layers on tcgen05 (see include/avc_b200.h: avc_lstm_seq).
//
// One time step is the GEMM  Z[B x 4H] = [x_t | h_{t-1}] . [W_ih | W_hh]^T  with the LSTM cell as its epilogue.
// Weight rows are gate-interleaved in groups of G hidden units, so a 128 x 4G accumulator tile holds all four gates
// of G units for 128 utterances: the epilogue thread that owns accumulator row b updates c[b, u] / h[b, u] for those G
// units without any cross-thread traffic.  h_{t-1} is read by TMA straight out of the output sequence [B][T][H] (a 3-D
// box {128 B, 1 frame, 128 utterances} at frame t-1), so there is no separate recurrent-state buffer.
//
// The step is bound by the shared-memory port (MMA operand reads + TMA fills, see DESIGN.md section 3), so the kernels
// minimise shared-memory bytes per MMA:
//   * CTA pairs (cta_group::2): a pair owns 256 utterances x 4G gate columns and each CTA stages only half of the W tile;
//   * split-bf16 ("fp32") mode loads {a_hi, a_lo, W_hi, W_lo} of a 64-channel chunk ONCE per stage and issues the
//     three products hi*hi, lo*hi, hi*lo from them (4 tiles instead of the 6 a K-concatenated GEMM would load);
//   * the W_hi and W_lo tiles of a stage are adjacent, so a_hi * [W_hi | W_lo] is ONE MMA of width 2 * BN into a
//     2 * BN-column accumulator (the a_hi tile is read once for both products) and a_lo * W_hi a second MMA of width BN
//     onto columns of the same gates; the cell warps add the two column blocks (SplitAcc below);
//   * "fp16x2" mode (fp16 activations, two-term fp16 weights) keeps only the wide MMA: {a, W_hi, W_lo} per stage, one
//     activation tile instead of two -- 9.6 K instead of 13.1 K cycles per frame for the H = 1024 recurrent part.
//
// Two kernels:
//   lstm_fused_kernel  (default) input projection and recurrence in one kernel, two TMEM accumulators: the x_t products
//                      of frame t+1 run while the cell update and the grid barrier of frame t are in flight
//   lstm_step_kernel   recurrence only, on a precomputed fp32 projection (xproj) -- small batches with wide inputs
// and two launch modes for each:
//   per-step    t_end = t_begin + 1, one launch per frame (stream order is the time dependency)
//   persistent  one cooperative launch for all frames; a barrier among the CTAs of a batch group separates frames
#include <cuda_bf16.h>
#include <cstdlib>
#include <type_traits>

#include "../../include/avc_b200.h"
#include "avc_host.h"
#include "avc_pipe.cuh"

namespace avc {

struct alignas(64) LstmParams {
  // One TMA op loads the hi AND lo tiles of a stage (the part is a tensor dimension): a TMA op costs ~100-170 cycles
  // of issue bandwidth whatever its size (scripts/ubench/tma_ops.cu), which is what bounds small-batch frames.
  CUtensorMap tmap_h;      // hseq as (H, B, part, T), box {kc, a_rows, PARTS, 1} -> [a_hi tile][a_lo tile]
  CUtensorMap tmap_w;      // w_hh as (H, 4H, part), box {kc, BN / CTAS, PARTS} -> [W_hi tile][W_lo tile]
  CUtensorMap tmap_x;      // xproj as (4H, T, B) fp32, box {32, 1, 128}
  CUtensorMap tmap_xi;     // fused input projection: input sequence as (C_in, B, part, T), box as tmap_h
  CUtensorMap tmap_wi;     // fused input projection: w_ih as (K_in, 4H, part), box as tmap_w
  const float* bias;       // fused input projection: b_ih + b_hh [4H], packed gate order
  int num_kx;              // fused input projection: k-blocks of the input part
  const float* xproj;
  void* hseq;
  float* hseq_f32;
  float* h_last;
  float* c_state;
  unsigned int* grid_barrier;
  long long* debug_clk;   // optional: 6 clock64 stamps per (frame, CTA)
  int B, T, H;
  int num_kb, kc_elems;
  int n_tiles;
  int t_begin, t_end;
  int a_rows;             // rows of an activation box: 128, or B rounded up to 8 when one CTA owns the whole batch
  int a_tile;             // bytes of one activation tile of a stage (a_rows * 128)
  int stage_bytes;        // {activation tile(s), W tile(s)}
  uint32_t stages;        // ring depth: as many stages as the shared-memory ring holds, at most kMaxStages
  uint32_t stage_tx;      // bytes one CTA's loads of a stage credit to the full barrier
};

// Accumulator layout of the split-bf16 mode.  Wide MMA (N = 2 * BN): B rows = this CTA's [W_hi tile ; W_lo tile], so with
// h = BN / CTAS gate columns per CTA the accumulator columns are, per CTA r of the pair, [hi*hi (h) | hi*lo (h)] at
// 2 * h * r.  Narrow MMA (N = BN, a_lo * W_hi): CTA r's h columns land at kLoOffset + h * r; with kLoOffset = h (pair) or 0
// (single CTA) every one of them falls on a block of the SAME gate columns, and z = first(c) + second(c).
template <int BN, int CTAS, bool SPLIT>
struct SplitAcc {
  static constexpr int kHalf = BN / CTAS;
  static constexpr int kCols = SPLIT ? 2 * BN : BN;                 // accumulator width in TMEM columns
  static constexpr int kLoOffset = (SPLIT && CTAS == 2) ? kHalf : 0;
  __device__ static constexpr int first(int c) { return (SPLIT && CTAS == 2 && c >= kHalf) ? c + kHalf : c; }
  __device__ static constexpr int second(int c) { return first(c) + kHalf; }
};

// The MMAs of one landed stage (activation tiles at `a_hi` / `a_lo`, W tile(s) at `w_hi`) into the accumulator at `acc`.
template <int BN, int MODE, int CTAS>
__device__ __forceinline__ void issue_stage(uint32_t a_hi, uint32_t a_lo, uint32_t w_hi, uint32_t acc, bool first) {
  constexpr bool BF16 = MODE != 0;
  if (MODE == 2) {
    issue_pair<2 * BN, BF16, CTAS>(a_hi, w_hi, acc, first);                                        // a_hi * [W_hi | W_lo]
    issue_pair<BN, BF16, CTAS>(a_lo, w_hi, acc + SplitAcc<BN, CTAS, true>::kLoOffset, false);                 // a_lo * W_hi
  } else if (MODE == 3) {
    issue_pair<2 * BN, BF16, CTAS>(a_hi, w_hi, acc, first, kIdescF16Xor);                          // a * [W_hi | W_lo], fp16
  } else {
    issue_pair<BN, BF16, CTAS>(a_hi, w_hi, acc, first);
  }
}

// Activation tile(s) of a stage: channels [kc0, kc0 + kc) of utterances [b0, b0 + a_rows) at frame t, both parts.
template <int CTAS>
__device__ __forceinline__ void load_act(void* dst, const CUtensorMap* map, uint64_t* bar, int kc0, int b0, int t) {
  if (CTAS == 2) tma_load_4d_2sm(dst, map, bar, kc0, b0, 0, t); else tma_load_4d(dst, map, bar, kc0, b0, 0, t);
}
// Weight tile(s) of a stage: channels [kc0, kc0 + kc) of rows [n, n + BN / CTAS), both parts.
template <int CTAS>
__device__ __forceinline__ void load_w(void* dst, const CUtensorMap* map, uint64_t* bar, int kc0, int n) {
  if (CTAS == 2) tma_load_3d_2sm(dst, map, bar, kc0, n, 0); else tma_load_3d(dst, map, bar, kc0, n, 0);
}

// Pre-activations (without bias / xproj) of hidden units j*8 .. j*8+7 of the tile for the four gates, from the
// accumulator row this thread owns; in split mode the sum of the two column blocks of SplitAcc.
template <class SA, int G>
__device__ __forceinline__ void load_gates(uint32_t lane_addr, int j, float (&z)[4][8]) {
  uint32_t a[4][8];
#pragma unroll
  for (int g = 0; g < 4; ++g) tmem_ld_32x8(lane_addr + SA::first(g * G + j * 8), a[g]);
  if (SA::kCols != 4 * G) {
    uint32_t b[4][8];
#pragma unroll
    for (int g = 0; g < 4; ++g) tmem_ld_32x8(lane_addr + SA::second(g * G + j * 8), b[g]);
    tmem_ld_wait();
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int e = 0; e < 8; ++e) z[g][e] = __uint_as_float(a[g][e]) + __uint_as_float(b[g][e]);
  } else {
    tmem_ld_wait();
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int e = 0; e < 8; ++e) z[g][e] = __uint_as_float(a[g][e]);
  }
}

// The same for a group of U (4 or 8) hidden units starting at unit j * U of the tile: tiles whose width is not a
// multiple of 8 units (G = 28: 37 tiles of H = 1024 fill all 148 SMs) are walked in groups of 4.
template <class SA, int G, int U>
__device__ __forceinline__ void load_gates_u(uint32_t lane_addr, int j, float (&z)[4][U]) {
  uint32_t a[4][U], b[4][U];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if constexpr (U == 8) tmem_ld_32x8(lane_addr + SA::first(g * G + j * U), a[g]);
    else tmem_ld_32x4(lane_addr + SA::first(g * G + j * U), a[g]);
  }
  if (SA::kCols != 4 * G) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if constexpr (U == 8) tmem_ld_32x8(lane_addr + SA::second(g * G + j * U), b[g]);
      else tmem_ld_32x4(lane_addr + SA::second(g * G + j * U), b[g]);
    }
    tmem_ld_wait();
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int e = 0; e < U; ++e) z[g][e] = __uint_as_float(a[g][e]) + __uint_as_float(b[g][e]);
  } else {
    tmem_ld_wait();
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int e = 0; e < U; ++e) z[g][e] = __uint_as_float(a[g][e]);
  }
}

// Stores of U (4 or 8) new hidden values of one cell thread: see store_h8.
template <int MODE, int U>
__device__ __forceinline__ void store_h_u(const LstmParams& p, long long row, int b, int t, int u, const float (&hn)[U]);

// Stores of one cell thread's 8 new hidden values (utterance row `row` = b*T + t, hidden units u..u+7): the recurrent
// operand in the layer's operand format, plus the optional exact fp32 copies.
template <int MODE>
__device__ __forceinline__ void store_h8(const LstmParams& p, long long row, int b, int t, int u, const float (&hn)[8]) {
  const long long hoff = row * p.H + u;
  if (MODE == 2) {
    float lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) lo[e] = hn[e] - __bfloat162float(__float2bfloat16_rn(hn[e]));
    __nv_bfloat16* hp = static_cast<__nv_bfloat16*>(p.hseq) + row * (2LL * p.H) + u;
    *reinterpret_cast<uint4*>(hp) = make_uint4(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]),
                                               pack_bf16(hn[4], hn[5]), pack_bf16(hn[6], hn[7]));
    *reinterpret_cast<uint4*>(hp + p.H) = make_uint4(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]),
                                                     pack_bf16(lo[4], lo[5]), pack_bf16(lo[6], lo[7]));
  } else if (MODE == 1) {
    uint4 pk = make_uint4(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]), pack_bf16(hn[4], hn[5]),
                          pack_bf16(hn[6], hn[7]));
    *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.hseq) + hoff) = pk;
  } else if (MODE == 3) {
    uint4 pk = make_uint4(pack_f16(hn[0], hn[1]), pack_f16(hn[2], hn[3]), pack_f16(hn[4], hn[5]),
                          pack_f16(hn[6], hn[7]));
    *reinterpret_cast<uint4*>(static_cast<__half*>(p.hseq) + hoff) = pk;
  } else {
    float* hp = static_cast<float*>(p.hseq) + hoff;
    *reinterpret_cast<float4*>(hp) =
        make_float4(round_tf32(hn[0]), round_tf32(hn[1]), round_tf32(hn[2]), round_tf32(hn[3]));
    *reinterpret_cast<float4*>(hp + 4) =
        make_float4(round_tf32(hn[4]), round_tf32(hn[5]), round_tf32(hn[6]), round_tf32(hn[7]));
  }
  if (p.hseq_f32) {
    float* hp = p.hseq_f32 + hoff;
    *reinterpret_cast<float4*>(hp) = make_float4(hn[0], hn[1], hn[2], hn[3]);
    *reinterpret_cast<float4*>(hp + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
  }
  if (p.h_last && t == p.T - 1) {
    float* hp = p.h_last + (long long)b * p.H + u;
    *reinterpret_cast<float4*>(hp) = make_float4(hn[0], hn[1], hn[2], hn[3]);
    *reinterpret_cast<float4*>(hp + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
  }
}

template <int MODE, int U>
__device__ __forceinline__ void store_h_u(const LstmParams& p, long long row, int b, int t, int u, const float (&hn)[U]) {
  if constexpr (U == 8) {
    store_h8<MODE>(p, row, b, t, u, hn);
  } else {
    static_assert(U == 4, "unit groups of 4 or 8");
    const long long hoff = row * p.H + u;
    if (MODE == 2) {
      float lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) lo[e] = hn[e] - __bfloat162float(__float2bfloat16_rn(hn[e]));
      __nv_bfloat16* hp = static_cast<__nv_bfloat16*>(p.hseq) + row * (2LL * p.H) + u;
      *reinterpret_cast<uint2*>(hp) = make_uint2(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]));
      *reinterpret_cast<uint2*>(hp + p.H) = make_uint2(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]));
    } else if (MODE == 1) {
      *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(p.hseq) + hoff) =
          make_uint2(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]));
    } else if (MODE == 3) {
      *reinterpret_cast<uint2*>(static_cast<__half*>(p.hseq) + hoff) =
          make_uint2(pack_f16(hn[0], hn[1]), pack_f16(hn[2], hn[3]));
    } else {
      *reinterpret_cast<float4*>(static_cast<float*>(p.hseq) + hoff) =
          make_float4(round_tf32(hn[0]), round_tf32(hn[1]), round_tf32(hn[2]), round_tf32(hn[3]));
    }
    if (p.hseq_f32) *reinterpret_cast<float4*>(p.hseq_f32 + hoff) = make_float4(hn[0], hn[1], hn[2], hn[3]);
    if (p.h_last && t == p.T - 1)
      *reinterpret_cast<float4*>(p.h_last + (long long)b * p.H + u) = make_float4(hn[0], hn[1], hn[2], hn[3]);
  }
}

// MODE: 0 = tf32, 1 = bf16, 2 = split bf16 (three bf16 products per fp32 product, operands staged once),
//       3 = fp16 activations x [W_hi | W_lo] fp16 weights (one wide MMA per stage: two products per fp32 product)
template <int BN, int MODE, int CTAS>
__global__ void __launch_bounds__(kNumThreads, 1) lstm_step_kernel(const __grid_constant__ LstmParams p) {
  constexpr int PARTS = MODE >= 2 ? 2 : 1;       // weight tiles per stage (ring sizing)
  constexpr int APARTS = MODE == 2 ? 2 : 1;      // activation tiles per stage
  constexpr int kXSlabs = BN / 32;                         // xproj tile = BN/32 swizzled slabs of 128 rows x 128 B
  constexpr int kXBytes = kXSlabs * kATileBytes;
  using SA = SplitAcc<BN, CTAS, MODE >= 2>;
  using C = PipeCfg<BN, CTAS, PARTS, false, kXBytes, 1, SA::kCols>;
  constexpr int G = BN / 4;
  extern __shared__ uint8_t smem_raw[];
  const PipeSmem s = carve_smem<C>(smem_raw);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = CTAS == 2 ? (int)cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit = blockIdx.x / CTAS;                       // one (pair of) CTA(s) per (m, n) tile
  const int n_tile = unit % p.n_tiles;
  const int m_tile = (unit / p.n_tiles) * CTAS + cta_rank;
  const int b0 = m_tile * kBlockM;
  const int n0 = n_tile * BN;
  const int nb0 = n0 + cta_rank * (BN / CTAS);              // first W_hh row staged by this CTA

  if (threadIdx.x == 0) {
    prefetch_tmap(&p.tmap_h);
    prefetch_tmap(&p.tmap_w);
    prefetch_tmap(&p.tmap_x);
  }
  const uint32_t tmem_base = pipe_setup<C>(s);

  RingState rs;              // producer and MMA issuer each keep their own copy (same sequence)
  uint32_t acc_phase = 0;    // epilogue: parity of tmem_full
  unsigned int sync_count = 0;
  int pre_issued = 0;        // producer: stages of the current frame whose W tiles are already in flight
  uint32_t epi_phase = 0;    // producer: parity of epi_done
  // cell warps: the running cell state lives in registers across frames; the xproj tile of each frame is fetched by
  // the producer thread with TMA into 128-byte-swizzled shared memory (a thread-per-row read of a swizzled slab is
  // bank-conflict free) while the MMAs of that frame run, so the cell warps issue no global loads.
  constexpr int NJ = (G / 8 + kEpiWarps / 4 - 1) / (kEpiWarps / 4);   // 8-unit groups per cell thread
  float4 cq[NJ][2];
  uint32_t x_phase = 0;

  for (int t = p.t_begin; t < p.t_end; ++t) {
    const bool has_mma = t > 0;   // h_{-1} = 0: the first frame has no recurrent term
    long long* dbg = p.debug_clk ? p.debug_clk + ((long long)t * gridDim.x + blockIdx.x) * 6 : nullptr;
    if (dbg && threadIdx.x == 0) dbg[0] = clock64();                       // frame start (after the grid barrier)
    if (warp == 0) {
      if (lane == 0) {
        // One stage = {h tile(s), W_hh tile(s)} of a 64/32-channel chunk.  The W_hh tiles do not depend on the previous
        // frame, so the first `pre` stages of frame t+1 get their W loads (and the full barrier's byte count) BEFORE
        // the grid barrier, while the cell epilogue of frame t is still running; only the h loads wait for it.
        auto issue = [&](int kb, int frame, bool want_w, bool want_h, uint32_t stage) {
          uint8_t* st = s.base + stage * p.stage_bytes;
          uint8_t* wst = st + APARTS * p.a_tile;
          const int kc0 = kb * p.kc_elems;
          if (want_w) {
            if (CTAS == 1 || leader) mbar_arrive_expect_tx(&s.full[stage], CTAS * p.stage_tx);
            load_w<CTAS>(wst, &p.tmap_w, &s.full[stage], kc0, nb0);
          }
          if (want_h) load_act<CTAS>(st, &p.tmap_h, &s.full[stage], kc0, b0, frame - 1);
        };
        auto issue_x = [&]() {     // this frame's xproj tile (independent of h): consumed by the cell warps
          mbar_arrive_expect_tx(s.extra_bar, kXBytes);
#pragma unroll
          for (int cc = 0; cc < kXSlabs; ++cc)
            tma_load_3d(s.extra + cc * kATileBytes, &p.tmap_x, s.extra_bar, n0 + cc * 32, t, b0);
        };
        if (!has_mma) issue_x();
        if (has_mma) {
          fence_proxy_async_global();   // h_{t-1} was written with generic stores (other CTAs / previous launch)
          RingState hs = rs;         // stages whose W tiles were pre-issued: add the h tiles
          for (int kb = 0; kb < pre_issued; ++kb) {
            issue(kb, t, false, true, hs.stage);
            hs.advance(p.stages);
          }
          for (int kb = 0; kb < pre_issued; ++kb) rs.advance(p.stages);
          issue_x();                 // after the h tiles of the first stages: those are on the critical path
          for (int kb = pre_issued; kb < p.num_kb; ++kb) {
            mbar_wait(&s.empty[rs.stage], rs.phase ^ 1u);
            issue(kb, t, true, true, rs.stage);
            rs.advance(p.stages);
          }
          pre_issued = 0;
        }
        if (t + 1 < p.t_end) {     // persistent mode: W tiles of the next frame's first stages
          RingState ws = rs;
          const int pre = p.num_kb < p.stages ? p.num_kb : p.stages;
          for (int kb = 0; kb < pre; ++kb) {
            mbar_wait(&s.empty[ws.stage], ws.phase ^ 1u);
            issue(kb, t + 1, true, false, ws.stage);
            ws.advance(p.stages);
          }
          pre_issued = pre;
          // the next frame's h tiles need every CTA's h_t: wait for this CTA's cell warps, then for the whole grid
          mbar_wait(s.epi_done, epi_phase);
          epi_phase ^= 1u;
          ++sync_count;
          // only the CTAs that own the same utterances (all n-tiles of this m tile / m pair) exchange h:
          // one counter per batch group (padded to its own 128-byte line)
          grid_arrive_wait(p.grid_barrier + 32 * (unit / p.n_tiles), sync_count * (unsigned)(p.n_tiles * CTAS));
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      if (lane == 0 && has_mma && leader) {
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&s.full[rs.stage], rs.phase);
          if (dbg && kb == 0) dbg[1] = clock64();                          // first stage landed
          tc_fence_after();
          const uint32_t a_hi = smem_u32(s.base + rs.stage * p.stage_bytes);
          const uint32_t w_hi = a_hi + APARTS * p.a_tile;
          issue_stage<BN, MODE, CTAS>(a_hi, a_hi + p.a_tile, w_hi, tmem_base, kb == 0);
          if (CTAS == 2) umma_commit_2sm(&s.empty[rs.stage], 0x3); else umma_commit(&s.empty[rs.stage]);
          rs.advance(p.stages);
        }
        if (CTAS == 2) umma_commit_2sm(s.tmem_full, 0x3); else umma_commit(s.tmem_full);
        if (dbg) dbg[2] = clock64();                                       // all MMAs issued
      }
      __syncwarp();
    } else {
      // ---------------- cell epilogue: thread owns utterance b; the two epilogue warps of a TMEM lane quarter
      // (warp_id % 4) take alternate groups of 8 hidden units of this tile
      const int q = warp & 3;
      const int half = (warp - 2) >> 2;
      const int b = b0 + q * 32 + lane;
      const bool valid = b < p.B;
      const int u0 = n_tile * G;
      const long long row = (long long)b * p.T + t;
      float* cp = p.c_state + (long long)b * p.H + u0;
      if (t == p.t_begin) {      // first frame of this launch
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
          const int j = half + jj * (kEpiWarps / 4);
          cq[jj][0] = cq[jj][1] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (valid && has_mma && j < G / 8) {      // per-step launches carry c through global memory
            cq[jj][0] = *reinterpret_cast<const float4*>(cp + j * 8);
            cq[jj][1] = *reinterpret_cast<const float4*>(cp + j * 8 + 4);
          }
        }
      }
      if (dbg && threadIdx.x == 64) dbg[3] = clock64();                    // xproj / c preloads issued
      if (has_mma) {
        mbar_wait(s.tmem_full, acc_phase);
        acc_phase ^= 1u;
        tc_fence_after();
      }
      mbar_wait(s.extra_bar, x_phase);                                     // xproj tile of this frame has landed
      x_phase ^= 1u;
      if (dbg && threadIdx.x == 64) dbg[4] = clock64();                    // accumulator ready
      const int xr = q * 32 + lane;                                        // this thread's row in the xproj tile
      const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll
      for (int jj = 0; jj < NJ; ++jj) {
        const int j = half + jj * (kEpiWarps / 4);
        if (j >= G / 8) break;
        float acc[4][8];
        if (has_mma) {
          load_gates<SA, G>(lane_addr, j, acc);
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[g][e] = 0.f;
        }
        if (valid) {
          float z[4][8];
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            // column g*G + j*8 of the tile: slab (col / 32), 16-byte chunk (col % 32) / 4, swizzled by row % 8
            const int col = g * G + j * 8;
            const uint8_t* slab = s.extra + (col >> 5) * kATileBytes + xr * 128;
            const int ch = (col & 31) >> 2;
            const float4 x0 = *reinterpret_cast<const float4*>(slab + ((ch ^ (xr & 7)) << 4));
            const float4 x1 = *reinterpret_cast<const float4*>(slab + (((ch + 1) ^ (xr & 7)) << 4));
            z[g][0] = acc[g][0] + x0.x;
            z[g][1] = acc[g][1] + x0.y;
            z[g][2] = acc[g][2] + x0.z;
            z[g][3] = acc[g][3] + x0.w;
            z[g][4] = acc[g][4] + x1.x;
            z[g][5] = acc[g][5] + x1.y;
            z[g][6] = acc[g][6] + x1.z;
            z[g][7] = acc[g][7] + x1.w;
          }
          const float4 c0 = cq[jj][0], c1 = cq[jj][1];
          const float cprev[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
          float cn[8], hn[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) lstm_cell(z[0][e], z[1][e], z[2][e], z[3][e], cprev[e], cn[e], hn[e]);
          cq[jj][0] = make_float4(cn[0], cn[1], cn[2], cn[3]);
          cq[jj][1] = make_float4(cn[4], cn[5], cn[6], cn[7]);
          if (t + 1 == p.t_end) {       // a later launch (per-step mode) resumes from global memory
            *reinterpret_cast<float4*>(cp + j * 8) = cq[jj][0];
            *reinterpret_cast<float4*>(cp + j * 8 + 4) = cq[jj][1];
          }
          store_h8<MODE>(p, row, b, t, u0 + j * 8, hn);
        }
      }
      fence_proxy_async_global();   // order the h stores before later async-proxy (TMA) reads
      tc_fence_before();         // ... and this warp's TMEM reads before the next frame's MMAs (via the barrier chain)
      __syncwarp();
      if (lane == 0) mbar_arrive(s.epi_done);
      if (dbg && threadIdx.x == 64) dbg[5] = clock64();                    // cell update done
    }
  }
  pipe_teardown<C>(tmem_base);
}


// ---------------------------------------------------------------------------------------------------------------
// Fused variant: the layer's input projection runs inside the recurrence kernel.
//   z_t = [x_t | h_{t-1}] . [W_ih | W_hh]^T + (b_ih + b_hh)
// The x_t part does not depend on the previous frame, so its MMAs (into the OTHER of two TMEM accumulators) run while
// the cell warps are still updating frame t-1 and while the grid barrier is in flight -- the tensor pipe no longer
// idles there -- and the fp32 xproj tensor (B*T*4H*4 bytes written and re-read per layer) never exists.
// Warp roles: 0 = producer of everything that is independent of the recurrence (x_t tiles, W_ih tiles, W_hh tiles);
// 1 = MMA issuer; 2..9 = cell warps; 10 = producer of the h_{t-1} tiles, which also owns the grid barrier.  Both
// producers walk the same ring in the same order: frame t = num_kx input stages, then (t > 0) num_kb recurrent stages.
constexpr int kFusedThreads = kNumThreads + 32;
constexpr int kBiasBytes = 1024;

template <int BN, int MODE, int CTAS>
__global__ void __launch_bounds__(kFusedThreads, 1) lstm_fused_kernel(const __grid_constant__ LstmParams p) {
  constexpr int PARTS = MODE >= 2 ? 2 : 1;       // weight tiles per stage (ring sizing)
  constexpr int APARTS = MODE == 2 ? 2 : 1;      // activation tiles per stage
  using SA = SplitAcc<BN, CTAS, MODE >= 2>;
  using C = PipeCfg<BN, CTAS, PARTS, false, kBiasBytes, 2, SA::kCols>;
  constexpr int G = BN / 4;
  static_assert(BN * 4 <= kBiasBytes - 16, "bias tile + the h_ready counter");
  extern __shared__ uint8_t smem_raw[];
  const PipeSmem s = carve_smem<C>(smem_raw);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = CTAS == 2 ? (int)cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit = blockIdx.x / CTAS;
  const int n_tile = unit % p.n_tiles;
  const int m_tile = (unit / p.n_tiles) * CTAS + cta_rank;
  const int b0 = m_tile * kBlockM;
  const int n0 = n_tile * BN;
  const int nb0 = n0 + cta_rank * (BN / CTAS);

  if (threadIdx.x == 0) {
    prefetch_tmap(&p.tmap_h);
    prefetch_tmap(&p.tmap_w);
    prefetch_tmap(&p.tmap_xi);
    prefetch_tmap(&p.tmap_wi);
  }
  float* sbias = reinterpret_cast<float*>(s.extra);
  // Recurrent stages whose slot the static producer has claimed (empty barrier observed, W tiles in flight).  The h
  // producer may not test the empty barriers itself: it skips the input stages, so it can be several ring rounds
  // ahead of the consumer, and an mbarrier parity wait only tells adjacent phases apart.
  uint32_t* h_ready = reinterpret_cast<uint32_t*>(s.extra + kBiasBytes - 16);
  if (threadIdx.x == 0) *h_ready = 0u;
  if (threadIdx.x >= 64 && threadIdx.x < 64 + BN) sbias[threadIdx.x - 64] = p.bias[n0 + threadIdx.x - 64];
  const uint32_t tmem_base = pipe_setup<C>(s);     // (its CTA / cluster barrier also publishes the bias tile)

  if (warp == 0) {
    if (lane == 0) {
      RingState rs;
      uint32_t h_claimed = 0;
      // one stage = {A tile(s), W tile(s)} of a 64/32-channel chunk; this thread credits the stage's full byte count
      // and loads everything except the h tiles
      auto stage_static = [&](const CUtensorMap* tw, int kb, const CUtensorMap* ta, int frame) {
        mbar_wait(&s.empty[rs.stage], rs.phase ^ 1u);
        uint8_t* st = s.base + rs.stage * p.stage_bytes;
        uint8_t* wst = st + APARTS * p.a_tile;
        const int kc0 = kb * p.kc_elems;
        if (CTAS == 1 || leader) mbar_arrive_expect_tx(&s.full[rs.stage], CTAS * p.stage_tx);
        load_w<CTAS>(wst, tw, &s.full[rs.stage], kc0, nb0);
        if (ta) load_act<CTAS>(st, ta, &s.full[rs.stage], kc0, b0, frame);
        if (!ta) {
          ++h_claimed;
          asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(smem_u32(h_ready)), "r"(h_claimed) : "memory");
        }
        rs.advance(p.stages);
      };
      for (int t = p.t_begin; t < p.t_end; ++t) {
        for (int kb = 0; kb < p.num_kx; ++kb) stage_static(&p.tmap_wi, kb, &p.tmap_xi, t);
        if (t > 0)
          for (int kb = 0; kb < p.num_kb; ++kb) stage_static(&p.tmap_w, kb, nullptr, 0);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      RingState rs;
      for (int t = p.t_begin; t < p.t_end; ++t) {
        long long* dbg = p.debug_clk ? p.debug_clk + ((long long)t * gridDim.x + blockIdx.x) * 8 : nullptr;
        const uint32_t acc = tmem_base + static_cast<uint32_t>((t & 1) * SA::kCols);
        const int total = p.num_kx + (t > 0 ? p.num_kb : 0);
        for (int i = 0; i < total; ++i) {
          if (dbg && i == p.num_kx) dbg[3] = clock64();                    // input part issued
          mbar_wait(&s.full[rs.stage], rs.phase);
          if (dbg && i == p.num_kx) dbg[1] = clock64();                    // first recurrent stage landed
          tc_fence_after();
          const uint32_t a_hi = smem_u32(s.base + rs.stage * p.stage_bytes);
          const uint32_t w_hi = a_hi + APARTS * p.a_tile;
          issue_stage<BN, MODE, CTAS>(a_hi, a_hi + p.a_tile, w_hi, acc, i == 0);
          if (CTAS == 2) umma_commit_2sm(&s.empty[rs.stage], 0x3); else umma_commit(&s.empty[rs.stage]);
          rs.advance(p.stages);
        }
        if (CTAS == 2) umma_commit_2sm(&s.tmem_full[t & 1], 0x3); else umma_commit(&s.tmem_full[t & 1]);
        if (dbg) dbg[2] = clock64();                                       // all MMAs of the frame issued
      }
    }
    __syncwarp();
  } else if (warp == 2 + kEpiWarps) {
    if (lane == 0) {
      RingState rs;
      uint32_t epi_phase = 0;
      uint32_t h_issued = 0;
      unsigned int sync_count = 0;
      for (int t = p.t_begin; t < p.t_end; ++t) {
        long long* dbg = p.debug_clk ? p.debug_clk + ((long long)t * gridDim.x + blockIdx.x) * 8 : nullptr;
        for (int kb = 0; kb < p.num_kx; ++kb) rs.advance(p.stages);
        if (t == 0) continue;
        if (t > p.t_begin) {
          // h_{t-1} comes from this launch: wait for this CTA's cell warps, then for every CTA that owns the same
          // utterances (all n-tiles of this m tile / m pair): one counter per batch group on its own 128-byte line
          ++sync_count;
          mbar_wait(s.epi_done, epi_phase);
          epi_phase ^= 1u;
          if (dbg) dbg[6] = clock64();                                     // this CTA's cell warps are done
          grid_arrive_wait(p.grid_barrier + 32 * (unit / p.n_tiles), sync_count * (unsigned)(p.n_tiles * CTAS),
                           dbg ? dbg + 7 : nullptr);
        }
        if (dbg) dbg[0] = clock64();                                       // barrier passed
        fence_proxy_async_global();   // h_{t-1} was written with generic stores (other CTAs / previous launch)
        for (int kb = 0; kb < p.num_kb; ++kb) {
          ++h_issued;
          {
            uint32_t seen;
            const long long t0 = clock64();
            do {
              asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(h_ready)) : "memory");
              if (seen < h_issued && clock64() - t0 > 4000000000LL) {
                printf("avc: h_ready timeout block %d seen %u want %u\n", (int)blockIdx.x, seen, h_issued);
                __trap();
              }
            } while (seen < h_issued);
          }
          uint8_t* st = s.base + rs.stage * p.stage_bytes;
          const int kc0 = kb * p.kc_elems;
          load_act<CTAS>(st, &p.tmap_h, &s.full[rs.stage], kc0, b0, t - 1);
          rs.advance(p.stages);
        }
      }
    }
    __syncwarp();
  } else {
    // ---------------- cell warps: thread owns utterance b; the two warps of a TMEM lane quarter take alternate groups
    // of U hidden units (8, or 4 when the tile width is not a multiple of 8 units); the running cell state stays in
    // registers across frames.  Units past H (the ragged last tile when G does not divide H) are never stored: their
    // weight rows and biases are zero padding.
    constexpr int U = G % 8 == 0 ? 8 : 4;
    constexpr int NG = G / U;
    static_assert(G % U == 0, "tile width must be a multiple of 4 hidden units");
    constexpr int NJ = (NG + kEpiWarps / 4 - 1) / (kEpiWarps / 4);
    float cq[NJ][U];
    uint32_t acc_phase = 0;      // bit i = parity of tmem_full[i]
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int b = b0 + q * 32 + lane;
    const bool valid = b < p.B;
    const int u0 = n_tile * G;
    float* cp = p.c_state + (long long)b * p.H + u0;
    for (int t = p.t_begin; t < p.t_end; ++t) {
      long long* dbg = p.debug_clk ? p.debug_clk + ((long long)t * gridDim.x + blockIdx.x) * 8 : nullptr;
      const long long row = (long long)b * p.T + t;
      if (t == p.t_begin) {
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
          const int j = half + jj * (kEpiWarps / 4);
#pragma unroll
          for (int e = 0; e < U; ++e) cq[jj][e] = 0.f;
          if (valid && t > 0 && j < NG && u0 + j * U < p.H) {      // per-step launches carry c through global memory
#pragma unroll
            for (int e = 0; e < U; e += 4) {
              const float4 c4 = *reinterpret_cast<const float4*>(cp + j * U + e);
              cq[jj][e] = c4.x; cq[jj][e + 1] = c4.y; cq[jj][e + 2] = c4.z; cq[jj][e + 3] = c4.w;
            }
          }
        }
      }
      const int buf = t & 1;
      mbar_wait(&s.tmem_full[buf], (acc_phase >> buf) & 1u);
      acc_phase ^= 1u << buf;
      tc_fence_after();
      if (dbg && threadIdx.x == 64) dbg[4] = clock64();                    // accumulator ready
      const uint32_t lane_addr =
          tmem_base + static_cast<uint32_t>(buf * SA::kCols) + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll
      for (int jj = 0; jj < NJ; ++jj) {
        const int j = half + jj * (kEpiWarps / 4);
        if (j >= NG) break;
        float acc[4][U];
        load_gates_u<SA, G, U>(lane_addr, j, acc);
        if (valid && u0 + j * U < p.H) {
          float z[4][U];
#pragma unroll
          for (int g = 0; g < 4; ++g) {
#pragma unroll
            for (int e = 0; e < U; e += 4) {
              const float4 x0 = *reinterpret_cast<const float4*>(sbias + g * G + j * U + e);       // broadcast reads
              z[g][e] = acc[g][e] + x0.x;
              z[g][e + 1] = acc[g][e + 1] + x0.y;
              z[g][e + 2] = acc[g][e + 2] + x0.z;
              z[g][e + 3] = acc[g][e + 3] + x0.w;
            }
          }
          float cn[U], hn[U];
#pragma unroll
          for (int e = 0; e < U; ++e) lstm_cell(z[0][e], z[1][e], z[2][e], z[3][e], cq[jj][e], cn[e], hn[e]);
#pragma unroll
          for (int e = 0; e < U; ++e) cq[jj][e] = cn[e];
          if (t + 1 == p.t_end) {       // a later launch (per-step mode) resumes from global memory
#pragma unroll
            for (int e = 0; e < U; e += 4)
              *reinterpret_cast<float4*>(cp + j * U + e) = make_float4(cn[e], cn[e + 1], cn[e + 2], cn[e + 3]);
          }
          store_h_u<MODE, U>(p, row, b, t, u0 + j * U, hn);
        }
      }
      fence_proxy_async_global();   // order the h stores before later async-proxy (TMA) reads
      tc_fence_before();            // ... and this warp's TMEM reads before the MMAs that reuse the accumulator
      __syncwarp();
      if (lane == 0) mbar_arrive(s.epi_done);
      if (dbg && threadIdx.x == 64) dbg[5] = clock64();                    // cell update done
    }
  }
  pipe_teardown<C>(tmem_base);
}

template <int BN, int MODE, int CTAS, bool FUSED>
static int run(LstmParams p, const avc_lstm_desc* d, int m_tiles, cudaStream_t stream) {
  auto kern = [] {      // (if constexpr: a tile width built for one kernel only must not instantiate the other)
    if constexpr (FUSED) return lstm_fused_kernel<BN, MODE, CTAS>;
    else return lstm_step_kernel<BN, MODE, CTAS>;
  }();
  constexpr int kAccCols = SplitAcc<BN, CTAS, MODE >= 2>::kCols;
  using C = std::conditional_t<FUSED, PipeCfg<BN, CTAS, MODE >= 2 ? 2 : 1, false, kBiasBytes, 2, kAccCols>,
                               PipeCfg<BN, CTAS, MODE >= 2 ? 2 : 1, false, BN / 32 * kATileBytes, 1, kAccCols>>;
  constexpr int kThreads = FUSED ? kFusedThreads : kNumThreads;
  // small batches shrink the stage (a_rows < 128): the same ring memory then holds more, shallower stages, which is what
  // a latency-bound frame wants (a TMA round trip costs ~3 K cycles whatever the tile size)
  const int fit = C::kStages * C::kStageBytes / p.stage_bytes;
  p.stages = (uint32_t)(fit < kMaxStages ? fit : kMaxStages);
  static PerDeviceOnce configured;
  if (configured.first_use()) {
    AVC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes));
  }
  const int grid = (m_tiles + CTAS - 1) / CTAS * CTAS * p.n_tiles;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CTAS > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CTAS;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (d->persistent) {
    AVC_REQUIRE(d->grid_barrier != nullptr, "avc_lstm_seq: persistent mode needs grid_barrier scratch");
    // AVC_LSTM_NO_COOP=1 (profiling aid): launch without the cooperative attribute.  Co-residency is then only
    // implied by the occupancy check below on an otherwise idle GPU; the bounded waits turn a violation into a trap.
    static const bool no_coop = getenv("AVC_LSTM_NO_COOP") != nullptr;
    if (!no_coop) {
      attr[na].id = cudaLaunchAttributeCooperative;
      attr[na].val.cooperative = 1;
      ++na;
    }
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  if (d->persistent) {
    int resident = 0;
    if (CTAS > 1) {
      int clusters = 0;
      AVC_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg));
      resident = clusters * CTAS;
    } else {
      int per_sm = 0;
      AVC_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, C::kSmemBytes));
      resident = per_sm * num_sms();
    }
    if (resident < grid) {   // distinct code: the caller may fall back to one launch per frame
      set_error("avc_lstm_seq: persistent grid %d does not fit (%d CTAs resident)", grid, resident);
      return AVC_ERR_NOT_RESIDENT;
    }
    AVC_REQUIRE((m_tiles + CTAS - 1) / CTAS <= 64, "avc_lstm_seq: at most 64 batch groups in persistent mode");
    AVC_CHECK_CUDA(cudaMemsetAsync(d->grid_barrier, 0, 64 * 32 * sizeof(unsigned int), stream));
    p.t_begin = 0;
    p.t_end = d->T;
    AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    count_launch();
  } else {
    for (int t = 0; t < d->T; ++t) {
      p.t_begin = t;
      p.t_end = t + 1;
      AVC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    }
    count_launch(d->T);
  }
  return 0;
}

static int lstm_cta_group() {
  static int v = 0;
  if (v == 0) {
    const char* e = getenv("AVC_LSTM_CTA_GROUP");
    v = (e && e[0] == '1') ? 1 : 2;
  }
  return v;
}

// h_last[b] = hseq_f32[b][lengths[b] - 1] (a padded batch).  The recurrence kernels keep their T - 1 store: a
// per-utterance comparison in their cell epilogue costs 4-9 registers in every instantiation (-Xptxas -v), so the
// variable-length form reads the exact fp32 copy of the sequence instead -- the same bits the in-kernel store writes.
__global__ void __launch_bounds__(256) gather_last_kernel(const float* __restrict__ hseq_f32, const int* __restrict__ lengths,
                                                          float* __restrict__ h_last, int T, int H) {
  const int b = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(hseq_f32 + ((long long)b * T + __ldg(lengths + b) - 1) * H);
  float4* dst = reinterpret_cast<float4*>(h_last + (long long)b * H);
  for (int i = threadIdx.x; i < H / 4; i += blockDim.x) dst[i] = src[i];
}

}  // namespace avc

extern "C" int avc_lstm_seq(const avc_lstm_desc* d, void* stream_v) {
  using namespace avc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  AVC_REQUIRE(d != nullptr, "avc_lstm_seq: null descriptor");
  if (d->lengths && d->h_last) {
    AVC_REQUIRE(d->hseq_f32 != nullptr, "avc_lstm_seq: lengths with h_last need hseq_f32 (h_last is read from it)");
    avc_lstm_desc full = *d;
    full.h_last = nullptr;
    full.lengths = nullptr;
    const int rc = avc_lstm_seq(&full, stream_v);
    if (rc != 0) return rc;
    gather_last_kernel<<<d->B, 256, 0, stream>>>(d->hseq_f32, d->lengths, d->h_last, d->T, d->H);
    AVC_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  AVC_REQUIRE(d->dtype >= AVC_DTYPE_TF32 && d->dtype <= AVC_DTYPE_F16, "avc_lstm_seq: bad dtype %d", d->dtype);
  AVC_REQUIRE(d->gate_group == 16 || d->gate_group == 28 || d->gate_group == 32, "avc_lstm_seq: gate_group %d (16, 28 or 32)",
              d->gate_group);
  const bool fused = d->xin != nullptr;
  // G = 28 (37 tiles of H = 1024: two batch groups x CTA pairs fill all 148 SMs) is built for the fused kernel only; its
  // last tile is ragged (H need not be a multiple of G: the packed weights carry zero rows for the missing units)
  AVC_REQUIRE(d->B > 0 && d->T > 0 && d->H > 0 && d->H % 4 == 0 && (d->H % d->gate_group == 0 || d->gate_group == 28),
              "avc_lstm_seq: bad shape B=%d T=%d H=%d", d->B, d->T, d->H);
  AVC_REQUIRE(d->gate_group != 28 || fused, "avc_lstm_seq: gate_group 28 needs the fused input projection (xin)");
  AVC_REQUIRE(d->w_hh && d->hseq && d->c_state, "avc_lstm_seq: missing buffer");
  AVC_REQUIRE(fused ? (d->w_ih && d->bias && !d->xproj) : d->xproj != nullptr,
              "avc_lstm_seq: give either xproj, or xin + w_ih + bias (fused input projection)");
  const int es = d->dtype == AVC_DTYPE_TF32 ? 4 : 2;
  const int kc = kRowBytes / es;
  AVC_REQUIRE(d->H % kc == 0, "avc_lstm_seq: H=%d must be a multiple of %d", d->H, kc);
  const int bn = 4 * d->gate_group;
  const bool split = d->dtype == AVC_DTYPE_BF16X3;                      // activations as [hi | lo]
  const bool w2 = split || d->dtype == AVC_DTYPE_F16;                   // weights as [w_hi | w_lo]
  const uint64_t H = (uint64_t)d->H;
  const int n_tiles = (d->H + d->gate_group - 1) / d->gate_group;
  const uint64_t w_rows = (uint64_t)n_tiles * bn;      // packed gate rows (4H, or more when the last tile is ragged)
  const uint64_t ld = split ? 2 * H : H;     // elements per row of hseq ([hi | lo] when split)
  const uint64_t ldw_hh = w2 ? 2 * H : H;    // elements per row of the packed W_hh
  const int m_tiles = (d->B + kBlockM - 1) / kBlockM;
  const int ctas = (m_tiles >= 2 && lstm_cta_group() == 2) ? 2 : 1;
  // A small batch owned by one CTA loads only its real rows (rounded up to 8): the MMA still spans 128 rows, but the
  // rows past the batch are never stored and every accumulator row depends on its own operand row only, so whatever
  // those shared-memory rows hold is harmless -- and the stage shrinks from 32 KB to a few KB of activations.
  const int a_rows = m_tiles == 1 ? (d->B + 7) / 8 * 8 : kBlockM;

  LstmParams p;
  memset(&p, 0, sizeof(p));
  const uint32_t parts = split ? 2 : 1, wparts = w2 ? 2 : 1;
  {
    const uint64_t dh[4] = {H, (uint64_t)d->B, parts, (uint64_t)d->T};
    const uint64_t sh[3] = {(uint64_t)d->T * ld * es, H * es, ld * es};
    const uint32_t bh[4] = {(uint32_t)kc, (uint32_t)a_rows, parts, 1};
    if (!encode_tmap_4d(&p.tmap_h, es, d->hseq, dh, sh, bh)) return -3;
    if (!encode_tmap_3d(&p.tmap_w, es, d->w_hh, H, w_rows, wparts, ldw_hh * es, H * es, kc, bn / ctas, wparts)) return -3;
  }
  if (fused) {
    // input sequence [B][T][xin_ld] holding xin_channels logical channels ([hi | lo] halves when split); channels past
    // xin_channels are zero-filled by TMA and meet zero columns of the K-padded w_ih
    const uint64_t cin = (uint64_t)d->xin_channels;
    AVC_REQUIRE(d->xin_channels > 0 && (cin * es) % 16 == 0, "avc_lstm_seq: xin_channels=%d", d->xin_channels);
    AVC_REQUIRE(d->xin_ld >= (long long)(split ? 2 * cin : cin), "avc_lstm_seq: xin_ld=%lld too small", d->xin_ld);
    p.num_kx = (int)((cin + kc - 1) / kc);
    const uint64_t kpad = (uint64_t)p.num_kx * kc;
    const uint64_t ldw = w2 ? 2 * kpad : kpad;
    const uint64_t dx[4] = {cin, (uint64_t)d->B, parts, (uint64_t)d->T};
    const uint64_t sx[3] = {(uint64_t)d->T * d->xin_ld * es, cin * es, (uint64_t)d->xin_ld * es};
    const uint32_t bx[4] = {(uint32_t)kc, (uint32_t)a_rows, parts, 1};
    if (!encode_tmap_4d(&p.tmap_xi, es, d->xin, dx, sx, bx)) return -3;
    if (!encode_tmap_3d(&p.tmap_wi, es, d->w_ih, kpad, w_rows, wparts, ldw * es, kpad * es, kc, bn / ctas, wparts)) return -3;
    p.bias = d->bias;
  } else {
    if (!encode_tmap_3d(&p.tmap_x, 4, d->xproj, 4 * H, (uint64_t)d->T, (uint64_t)d->B, 4 * H * 4,
                        (uint64_t)d->T * 4 * H * 4, 32, 1, kBlockM))
      return -3;
  }
  p.xproj = d->xproj;
  p.hseq = d->hseq;
  p.hseq_f32 = d->hseq_f32;
  p.h_last = d->h_last;
  p.c_state = d->c_state;
  p.grid_barrier = d->grid_barrier;
  p.debug_clk = d->debug_clk;
  p.B = d->B;
  p.T = d->T;
  p.H = d->H;
  p.kc_elems = kc;
  p.num_kb = d->H / kc;
  p.n_tiles = n_tiles;
  p.a_rows = a_rows;
  p.a_tile = a_rows * kRowBytes;
  p.stage_bytes = (int)parts * p.a_tile + (int)wparts * (bn / ctas * kRowBytes);
  p.stage_tx = (uint32_t)p.stage_bytes;
#define AVC_LSTM_DISPATCH3(BN_, MODE_, CTAS_) \
  return fused ? run<BN_, MODE_, CTAS_, true>(p, d, m_tiles, stream) : run<BN_, MODE_, CTAS_, false>(p, d, m_tiles, stream);
#define AVC_LSTM_DISPATCH2(BN_, MODE_) \
  if (ctas == 2) { AVC_LSTM_DISPATCH3(BN_, MODE_, 2) } else { AVC_LSTM_DISPATCH3(BN_, MODE_, 1) }
#define AVC_LSTM_DISPATCH(BN_)                           \
  switch (d->dtype) {                                    \
    case AVC_DTYPE_TF32: AVC_LSTM_DISPATCH2(BN_, 0)      \
    case AVC_DTYPE_BF16: AVC_LSTM_DISPATCH2(BN_, 1)      \
    case AVC_DTYPE_F16: AVC_LSTM_DISPATCH2(BN_, 3)       \
    default: AVC_LSTM_DISPATCH2(BN_, 2)                  \
  }
  if (bn == 112) {      // fused kernel only, 16-bit two-term precisions, CTA pairs (the full-batch configuration it exists for)
    AVC_REQUIRE(ctas == 2 && (d->dtype == AVC_DTYPE_F16 || d->dtype == AVC_DTYPE_BF16X3),
                "avc_lstm_seq: gate_group 28 needs B > 128 and the fp16x2 / split precision");
    if (d->dtype == AVC_DTYPE_F16) return run<112, 3, 2, true>(p, d, m_tiles, stream);
    return run<112, 2, 2, true>(p, d, m_tiles, stream);
  }
  switch (bn) {
    case 64: AVC_LSTM_DISPATCH(64)
    default: AVC_LSTM_DISPATCH(128)
  }
#undef AVC_LSTM_DISPATCH
#undef AVC_LSTM_DISPATCH3
#undef AVC_LSTM_DISPATCH2
}
