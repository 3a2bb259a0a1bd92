// The TMA -> shared memory -> tcgen05.mma pipeline shared by the convolution/GEMM kernel and the
// LSTM step kernel.  One CTA computes a 128 x BN fp32 accumulator tile in tensor memory:
//   warp 0 (one lane)  : TMA producer, ring of STAGES {A 128x128B, B BNx128B} tiles, 128-byte swizzle
//   warp 1 (one lane)  : tcgen05.mma issuer, 4 MMAs (32 bytes of K each) per k-block
//   warps 2..5         : epilogue (TMEM -> registers -> global)
// K is consumed in k-blocks of 128 bytes per row: 32 TF32 or 64 bf16 elements.
#pragma once
#include "avc_ptx.cuh"

namespace avc {

constexpr int kBlockM = 128;
constexpr int kRowBytes = 128;                 // one swizzle row = one k-block of one row
constexpr int kATileBytes = kBlockM * kRowBytes;  // 16 KB
constexpr int kMaxStages = 8;                   // barrier slots reserved for the ring (a kernel may run fewer stages)
constexpr int kEpiWarps = 8;                   // two epilogue warps per TMEM lane quarter (= per SM sub-partition)
constexpr int kNumThreads = 64 + 32 * kEpiWarps;   // TMA warp + MMA warp + epilogue warps
constexpr int kSmemBudget = 186 * 1024;
constexpr int kStagingLd = 36;                  // floats per staged row: 32 + 4 pad keeps 16-byte accesses conflict free
constexpr int kStagingBytes = kEpiWarps * 32 * kStagingLd * 4;   // one 32 x 32 transpose tile per epilogue warp

// CTAS = 1: one CTA owns a 128 x BN tile.  CTAS = 2: a CTA pair (cta_group::2) owns a 256 x BN tile; each CTA stages its
// own 128 A rows and BN/2 of the B rows, and the leader CTA's MMA thread issues for both.
// PARTS = 1: a stage holds one {A, B} operand pair.  PARTS = 2 (split-bf16 recurrence): a stage holds {A_hi, A_lo,
// B_hi, B_lo} of one 64-channel chunk, from which the three products hi*hi, lo*hi, hi*lo are issued.
// STAGING: reserve the epilogue's per-warp transpose tiles.
// EXTRA: bytes of kernel-specific shared memory (1024-byte aligned) placed after the stages, with one extra mbarrier.
// ACC: accumulator buffers in tensor memory (2 = the epilogue of tile i overlaps the MMAs of tile i+1).
// ACCW: tensor-memory columns per accumulator buffer (BN, or 2 * BN for the split recurrence's wide accumulator).
template <int BN, int CTAS = 1, int PARTS = 1, bool STAGING = true, int EXTRA = 0, int ACC = 1, int ACCW = BN>
struct PipeCfg {
  static constexpr int kAcc = ACC;
  static constexpr int kCtas = CTAS;
  static constexpr int kParts = PARTS;
  static constexpr int kBTileBytes = BN / CTAS * kRowBytes;
  static constexpr int kStageBytes = PARTS * (kATileBytes + kBTileBytes);
  static constexpr int kBudget = (STAGING ? kSmemBudget : kSmemBudget + kStagingBytes + 8 * 1024) - EXTRA;
  static constexpr int kStages = (kBudget / kStageBytes) > kMaxStages ? kMaxStages : (kBudget / kStageBytes);
  // per-epilogue-warp staging tile used to transpose 32 rows x 32 columns so that global stores are coalesced
  static constexpr int kExtraOffset = kStages * kStageBytes;
  static constexpr int kStagingOffset = kExtraOffset + EXTRA;
  static constexpr int kBarOffset = kStagingOffset + (STAGING ? kStagingBytes : 0);
  // full[kMaxStages], empty[kMaxStages], tmem_full[2], tmem_empty[2], extra barrier, epilogue-done barrier, TMEM address word
  static constexpr int kSmemBytes = kBarOffset + (2 * kMaxStages + 6) * 8 + 16 + 1024 /* alignment slack */;
  static constexpr int kAccCols = ACCW;
  static constexpr uint32_t pow2_at_least(uint32_t v) { uint32_t r = 32; while (r < v) r <<= 1; return r; }
  static constexpr uint32_t kTmemCols = pow2_at_least(ACCW * ACC);      // allocations are powers of two >= 32
  static_assert(kTmemCols <= 512, "TMEM columns: at most 512");
  static_assert(kStages >= 2, "pipeline needs at least two stages");
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget exceeded");
};

struct PipeSmem {
  uint8_t* base;        // 1024-byte aligned
  float* staging;
  uint64_t* full;
  uint64_t* empty;
  uint64_t* tmem_full;    // [2]
  uint64_t* tmem_empty;   // [2]
  uint64_t* extra_bar;
  uint64_t* epi_done;     // count kEpiWarps: every epilogue warp of THIS CTA has finished its part
  uint8_t* extra;
  uint32_t* tmem_ptr;
};

template <class C>
__device__ __forceinline__ PipeSmem carve_smem(uint8_t* raw) {
  PipeSmem s;
  const uint32_t addr = smem_u32(raw);
  s.base = raw + ((1024u - (addr & 1023u)) & 1023u);
  s.staging = reinterpret_cast<float*>(s.base + C::kStagingOffset);
  s.full = reinterpret_cast<uint64_t*>(s.base + C::kBarOffset);
  s.empty = s.full + kMaxStages;
  s.tmem_full = s.empty + kMaxStages;
  s.tmem_empty = s.tmem_full + 2;
  s.extra_bar = s.tmem_empty + 2;
  s.epi_done = s.extra_bar + 1;
  s.extra = s.base + C::kExtraOffset;
  s.tmem_ptr = reinterpret_cast<uint32_t*>(s.epi_done + 1);
  return s;
}

// Barrier init (thread 0) + TMEM allocation (warp 1) + CTA / cluster sync.  Returns the TMEM base address.
template <class C>
__device__ __forceinline__ uint32_t pipe_setup(const PipeSmem& s) {
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(&s.full[i], 1);
      mbar_init(&s.empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.tmem_full[i], 1);
      mbar_init(&s.tmem_empty[i], C::kCtas * kEpiWarps);   // one arrival per epilogue warp of every CTA of the pair
    }
    mbar_init(s.extra_bar, 1);
    mbar_init(s.epi_done, kEpiWarps);
    fence_mbar_init();
  }
  if (warp == 1) {
    if (C::kCtas == 2) {
      tmem_alloc_2sm(s.tmem_ptr, C::kTmemCols);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(s.tmem_ptr, C::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (C::kCtas == 2)
    cluster_sync_all();   // the peer's TMA credits bytes to the leader's barriers: inits must be visible cluster-wide
  else
    __syncthreads();
  tc_fence_after();
  return *reinterpret_cast<volatile uint32_t*>(s.tmem_ptr);
}

template <class C>
__device__ __forceinline__ void pipe_teardown(uint32_t tmem_base) {
  __syncwarp();
  tc_fence_before();
  if (C::kCtas == 2)
    cluster_sync_all();   // neither CTA may free TMEM / exit while the pair's MMAs or multicast arrivals are pending
  else
    __syncthreads();
  if ((threadIdx.x >> 5) == 1) {
    tc_fence_after();
    if (C::kCtas == 2)
      tmem_dealloc_2sm(tmem_base, C::kTmemCols);
    else
      tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

struct RingState {
  uint32_t stage = 0;
  uint32_t phase = 0;
  template <int STAGES>
  __device__ __forceinline__ void advance() {
    if (++stage == STAGES) {
      stage = 0;
      phase ^= 1u;
    }
  }
  __device__ __forceinline__ void advance(uint32_t stages) {   // ring depth chosen at launch
    if (++stage == stages) {
      stage = 0;
      phase ^= 1u;
    }
  }
};

// Four MMAs (32 bytes of K each) over one 128-byte-wide operand pair: D (+)= A[128*CTAS x 128B] . B[BN x 128B]^T.
// `fmt_xor` = kIdescF16Xor turns the 16-bit operand format from bf16 into fp16 (same instruction, same tiles).
constexpr uint32_t kIdescF16Xor = (1u << 7) | (1u << 10);
template <int BN, bool BF16, int CTAS>
__device__ __forceinline__ void issue_pair(uint32_t a_addr, uint32_t b_addr, uint32_t tmem_acc, bool first,
                                           uint32_t fmt_xor = 0) {
  const uint32_t idesc = umma_idesc(kBlockM * CTAS, BN, !BF16) ^ fmt_xor;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint64_t adesc = umma_desc_sw128(a_addr + k * 32);
    const uint64_t bdesc = umma_desc_sw128(b_addr + k * 32);
    const uint32_t acc = (first && k == 0) ? 0u : 1u;
    if (CTAS == 2) {
      if (BF16)
        umma_bf16_2sm(tmem_acc, adesc, bdesc, idesc, acc);
      else
        umma_tf32_2sm(tmem_acc, adesc, bdesc, idesc, acc);
    } else {
      if (BF16)
        umma_bf16(tmem_acc, adesc, bdesc, idesc, acc);
      else
        umma_tf32(tmem_acc, adesc, bdesc, idesc, acc);
    }
  }
}

// MMA issue for one k-block that has landed in `stage` of a PARTS = 1 pipeline.
template <int BN, bool BF16, int CTAS = 1>
__device__ __forceinline__ void issue_kblock(const PipeSmem& s, uint32_t stage, uint32_t tmem_acc, bool first,
                                             uint32_t fmt_xor = 0) {
  using C = PipeCfg<BN, CTAS>;
  const uint32_t a_addr = smem_u32(s.base + stage * C::kStageBytes);
  issue_pair<BN, BF16, CTAS>(a_addr, a_addr + kATileBytes, tmem_acc, first, fmt_xor);
}

// Grid barrier executed by ONE thread per CTA (the TMA producer): everything that must be ordered before it in this CTA
// has already synchronised with this thread through the epi_done mbarrier.
__device__ __forceinline__ void grid_arrive_wait(unsigned int* bar, unsigned int target, long long* stamp = nullptr) {
  // release: everything this thread has observed (the cell warps' h stores, via epi_done) becomes visible to whoever
  // acquires the counter; the acquire load orders the TMA issue that follows.
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
  const long long t0 = clock64();
  if (stamp) *stamp = t0;                                                  // arrival issued (after the release fence)
  unsigned int seen;
  do {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(bar) : "memory");
    if (seen < target && clock64() - t0 > 4000000000LL) {
      printf("avc: grid barrier timeout block %d seen %u target %u\n", (int)blockIdx.x, seen, target);
      __trap();
    }
  } while (seen < target);
}

// Frame of utterance b whose h goes to h_last: lengths[b] - 1 of a padded batch, else T - 1.  The length is read where it
// is compared, with a volatile load the compiler can neither hoist into a register held across the frame loop nor
// speculate (the weight-stationary kernel keeps its register allocation with it, -Xptxas -v).
__device__ __forceinline__ bool is_last_frame(const int* lengths, int b, int t, int T) {
  if (!lengths) return t == T - 1;
  int len;
  asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(len) : "l"(lengths + b));
  return t == len - 1;
}

// Utterance of `tile` in the compacted tile space of a padded batch: the b with tile_start[b] <= tile < tile_start[b + 1]
// (tile_start [B + 1] is a strictly increasing prefix table, every utterance has at least one tile).
__device__ __forceinline__ int ragged_tile_utt(const int* __restrict__ tile_start, int B, int tile) {
  int lo = 0, hi = B;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(tile_start + mid) <= tile) lo = mid;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
// tanh with ~1e-7 absolute error (tanh.approx is only good to 2^-11, too coarse for a 1e-3 end-to-end gate).
__device__ __forceinline__ float tanh_fast(float x) {
  const float e = __expf(-2.0f * fabsf(x));
  const float r = __fdividef(1.0f - e, 1.0f + e);
  return copysignf(r, x);
}
// LSTM cell with 7 instead of 10 MUFU operations per hidden unit: the three sigmoids and tanh(g) share ONE reciprocal
// (s_i = N_i / D with D = (1+e_i)(1+e_f)(1+e_o)(1+e_g)); inputs are clamped to +-25 so D stays below 2^110.
__device__ __forceinline__ void lstm_cell(float zi, float zf, float zg, float zo, float c_prev, float& c_new,
                                          float& h_new) {
  const float ei = __expf(-fminf(fmaxf(zi, -25.0f), 25.0f));
  const float ef = __expf(-fminf(fmaxf(zf, -25.0f), 25.0f));
  const float eo = __expf(-fminf(fmaxf(zo, -25.0f), 25.0f));
  const float eg = __expf(-2.0f * fabsf(zg));                  // in (0, 1]
  const float di = 1.0f + ei, df = 1.0f + ef, dq = 1.0f + eo, dg = 1.0f + eg;
  const float dif = di * df, dog = dq * dg;
  const float r = __fdividef(1.0f, dif * dog);
  const float si = r * df * dog;                               // 1 / (1 + e_i)
  const float sf = r * di * dog;
  const float so = r * dif * dg;
  const float tg = copysignf((1.0f - eg) * (r * dif * dq), zg);   // tanh(z_g)
  c_new = sf * c_prev + si * tg;
  h_new = so * tanh_fast(c_new);
}

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// fp16 stores saturate at +-65504 instead of producing inf (an out-of-range activation then costs accuracy, not a
// NaN-poisoned utterance; values on this path are O(1..100))
__device__ __forceinline__ float sat_f16(float v) { return fminf(fmaxf(v, -65504.0f), 65504.0f); }
// two floats -> packed fp16 pair with saturation, ONE instruction (F2FP.SATFINITE.F16.F32.PACK_AB); `lo` lands in the low half
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// second term of the two-term fp16 form v ~ hi + lo, hi = fp16(v): what fp16(v) lost (exact in fp32, ~2^-22 relative after
// its own rounding; values below fp16's subnormal step flush towards zero, which costs < 6e-8 absolute)
__device__ __forceinline__ float f16_lo(float v) {
  const float s = sat_f16(v);
  return s - __half2float(__float2half_rn(s));
}
// Cheaper two-term split for the fused ResnetBlock epilogues (6 instructions for two values): hi = v with the 13 low
// mantissa bits cleared -- exactly representable in fp16 over its normal range, so the pack below is exact -- and
// lo = v - hi, exact in fp32, < 2^-10 |v|, rounded to fp16 by its own pack: hi + lo = v to ~2^-21.  (hi is truncated, not
// rounded, so it is NOT fp16(v); every consumer reads hi + lo.)  Out-of-range values saturate in the packs.
__device__ __forceinline__ void split_f16_pair_trunc(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const float h0 = __uint_as_float(__float_as_uint(v0) & 0xFFFFE000u);
  const float h1 = __uint_as_float(__float_as_uint(v1) & 0xFFFFE000u);
  hi = pack_f16(h0, h1);
  lo = pack_f16(v0 - h0, v1 - h1);
}
// (v0, v1) -> packed hi pair and packed lo pair of the two-term form (8 instructions for two values)
__device__ __forceinline__ void split_f16_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  hi = pack_f16(v0, v1);
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  lo = pack_f16(sat_f16(v0) - h.x, sat_f16(v1) - h.y);
}

}  // namespace avc
