// Host-side helpers shared by the translation units of libavc_b200.so: error text, launch counter,
// TMA tensor-map encoding through the driver entry point (no link-time dependency on libcuda, so the
// library also loads on a box without a GPU driver).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

namespace avc {

void set_error(const char* fmt, ...);
void count_launch(long long n = 1);

// 3-D tiled tensor map over a [d2][d1][d0] array (d0 contiguous), 128-byte swizzle, zero OOB fill.
// elem_bytes = 4 (fp32 read as TF32) or 2 (bf16).  Box = {box0, box1, box2} elements; box0*elem_bytes == 128.
bool encode_tmap_3d(CUtensorMap* map, int elem_bytes, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                    uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1, uint32_t box2);
// 4-D variant: dims d[0] (contiguous) .. d[3], stride_bytes[i] = byte stride of dim i + 1, box b[0..3].
bool encode_tmap_4d(CUtensorMap* map, int elem_bytes, const void* base, const uint64_t (&d)[4],
                    const uint64_t (&stride_bytes)[3], const uint32_t (&b)[4]);
// 2-D variant over [d1][d0].
bool encode_tmap_2d(CUtensorMap* map, int elem_bytes, const void* base, uint64_t d0, uint64_t d1,
                    uint64_t stride1_bytes, uint32_t box0, uint32_t box1);

int num_sms();   // of the CURRENT device (cached per device)

// Launch set-up of a persistent kernel whose CTAs wait on each other through a grid barrier: the cluster attribute
// (cluster > 1) and the cooperative attribute go into `attr` / `cfg`, then the occupancy query.  A grid that cannot be
// resident at once returns AVC_ERR_NOT_RESIDENT with the error text set, before anything is launched, so the caller may
// fall back.  AVC_LSTM_NO_COOP set (profiling aid: a profiler cannot replay a cooperative launch) drops the cooperative
// attribute: co-residency then rests on this occupancy check on an otherwise idle GPU, and the kernels' bounded waits
// turn a violation into a trap.  Returns 0, AVC_ERR_NOT_RESIDENT, or -2 on a CUDA error.
int persistent_launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute (&attr)[2], const void* kern, int cluster,
                             const char* name);

// Per-device "already configured" flag for a kernel's cudaFuncSetAttribute: function attributes are per device, so a
// process that drives several GPUs must set them once on each.  One instance per kernel instantiation (a function-local
// static at the launch site); `first_use()` returns true exactly once per (instance, current device).
struct PerDeviceOnce {
  static constexpr int kMaxDevices = 64;
  bool done[kMaxDevices] = {};
  bool first_use() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return true;   // unknown: always configure
    if (done[dev]) return false;
    done[dev] = true;
    return true;
  }
};

#define AVC_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      avc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return -2;                                                                          \
    }                                                                                     \
  } while (0)

#define AVC_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      avc::set_error(__VA_ARGS__);    \
      return -1;                      \
    }                                 \
  } while (0)

}  // namespace avc
