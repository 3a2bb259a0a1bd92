// Host-side plumbing of libavc_b200.so (see avc_host.h).
#include "avc_host.h"

#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/avc_b200.h"

namespace avc {

static thread_local char g_error[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

void count_launch(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static bool encode(CUtensorMap* map, int elem_bytes, const void* base, int rank, const cuuint64_t* dims,
                   const cuuint64_t* strides, const cuuint32_t* box) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return false;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15u) != 0) {
    set_error("tensor map base %p is not 16-byte aligned", base);
    return false;
  }
  for (int i = 0; i + 1 < rank; ++i) {
    if (strides[i] % 16 != 0) {
      set_error("tensor map stride %d = %llu bytes is not a multiple of 16", i, (unsigned long long)strides[i]);
      return false;
    }
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUtensorMapDataType dt = elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = fn(map, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu,%llu box %u,%u,%u)", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
    return false;
  }
  return true;
}

bool encode_tmap_3d(CUtensorMap* map, int elem_bytes, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                    uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1, uint32_t box2) {
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  return encode(map, elem_bytes, base, 3, dims, strides, box);
}

bool encode_tmap_4d(CUtensorMap* map, int elem_bytes, const void* base, const uint64_t (&d)[4],
                    const uint64_t (&stride_bytes)[3], const uint32_t (&b)[4]) {
  cuuint64_t dims[4] = {d[0], d[1], d[2], d[3]};
  cuuint64_t strides[3] = {stride_bytes[0], stride_bytes[1], stride_bytes[2]};
  cuuint32_t box[4] = {b[0], b[1], b[2], b[3]};
  return encode(map, elem_bytes, base, 4, dims, strides, box);
}

bool encode_tmap_2d(CUtensorMap* map, int elem_bytes, const void* base, uint64_t d0, uint64_t d1,
                    uint64_t stride1_bytes, uint32_t box0, uint32_t box1) {
  cuuint64_t dims[2] = {d0, d1};
  cuuint64_t strides[1] = {stride1_bytes};
  cuuint32_t box[2] = {box0, box1};
  return encode(map, elem_bytes, base, 2, dims, strides, box);
}

int num_sms() {
  static int n[PerDeviceOnce::kMaxDevices] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= PerDeviceOnce::kMaxDevices) return 148;
  if (n[dev] == 0 && cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n[dev] = 148;
  return n[dev];
}

int persistent_launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute (&attr)[2], const void* kern, int cluster,
                             const char* name) {
  static const bool no_coop = getenv("AVC_LSTM_NO_COOP") != nullptr;
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (!no_coop) {
    attr[na].id = cudaLaunchAttributeCooperative;
    attr[na].val.cooperative = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  int resident = 0;
  if (cluster > 1) {
    int clusters = 0;
    AVC_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg));
    resident = clusters * cluster;
  } else {
    int per_sm = 0;
    AVC_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, (int)cfg.blockDim.x, cfg.dynamicSmemBytes));
    resident = per_sm * num_sms();
  }
  const int grid = (int)cfg.gridDim.x;
  if (resident < grid) {
    set_error("%s: persistent grid %d does not fit (%d CTAs resident)", name, grid, resident);
    return AVC_ERR_NOT_RESIDENT;
  }
  return 0;
}

}  // namespace avc

extern "C" int avc_version(void) { return 100; }
extern "C" const char* avc_last_error(void) { return avc::g_error; }
extern "C" long long avc_launch_count(void) { return avc::g_launches.load(std::memory_order_relaxed); }
