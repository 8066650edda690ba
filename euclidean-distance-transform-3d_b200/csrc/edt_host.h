// edt_host.h -- declarations shared by the host-side translation units of libedt_b200.so.
//
// The library is compiled as five translation units so that the kernel templates build in
// parallel: edt_capi.cu (C ABI, staging, caches) and edt_passes_b{1,2,4,8}.cu (the axis-pass
// launchers of edt_passes.cuh instantiated for one label width each).
#pragma once
#include "../../include/edt_b200.h"
#include "edt_kernels.cuh"

#include <cstdint>
#include <mutex>

namespace edtb200 {
namespace host {

// Sets the calling thread's error message (edtb200_last_error) and returns `code`.
int fail(int code, const char* fmt, ...);

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess)                                                                     \
      return ::edtb200::host::fail(e__ == cudaErrorMemoryAllocation ? EDTB200_ENOMEM : EDTB200_ECUDA, \
                                   "%s failed: %s", #expr, cudaGetErrorString(e__));            \
  } while (0)

// cuTensorMapEncodeTiled, fetched through the runtime so that libcuda is not a link-time
// dependency (the library must load on machines without a driver, e.g. for the build check).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder();

// Per-device cached state.  `lock` guards the mutable members (buffers, tables, streams); it is
// held only while they are looked up or changed, never across a whole transform.  `host_call`
// serialises the calls that stage HOST buffers through this device's cached device buffers --
// calls on different devices run concurrently.
struct DeviceCache {
  std::mutex lock;
  std::mutex host_call;
  void* labels = nullptr;
  size_t labels_bytes = 0;
  float* dist = nullptr;
  size_t dist_bytes = 0;
  cudaStream_t stream = nullptr;
  // second slot + copy streams + events of edtb200_transform_batch (slot 0 is labels / dist above)
  void* labels2 = nullptr;
  size_t labels2_bytes = 0;
  float* dist2 = nullptr;
  size_t dist2_bytes = 0;
  cudaStream_t stream_up = nullptr, stream_down = nullptr;
  cudaEvent_t ev_up[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_down[2] = {nullptr, nullptr};
  // step tables T[k] of the first-axis pass, keyed by the weight's bits (see step_table_kernel).
  // A table remembers the streams that used it (one event each) so that it can be retired
  // without a device-wide synchronisation when the cache is full.
  struct Table {
    float* data = nullptr; int count = 0; uint32_t wbits = 0; uint64_t stamp = 0;
    cudaEvent_t ready = nullptr; cudaStream_t built_on = nullptr;
    static constexpr int kUsers = 4;
    cudaStream_t user[kUsers] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t used[kUsers] = {nullptr, nullptr, nullptr, nullptr};
    bool user_set[kUsers] = {false, false, false, false};
    bool many_users = false;
  };
  static constexpr int kTables = 16;
  Table tables[kTables];
  uint64_t table_clock = 0;
  cudaMemPool_t pool = nullptr;        // private pool of the stream-ordered scratch allocations
  // run statistic of the first-axis pass (see RunStat): device counters + a mapped host word pair
  unsigned long long* stat_counter = nullptr;
  unsigned int* stat_ticket = nullptr;
  volatile unsigned long long* stat_publish_host = nullptr;
  unsigned long long* stat_publish_dev = nullptr;
  int sm_count = 0;
  int max_smem_optin = 0;
  bool probed = false;
};

// Stream-ordered scratch from the device's private pool (never the process-wide default pool).
cudaError_t scratch_alloc(DeviceCache& dc, void** p, size_t bytes, cudaStream_t stream);

// Device table T[0..count) for weight w, cached per device.
int step_table(DeviceCache& dc, float w, int count, cudaStream_t stream, const float** out);
// To be called once the kernel reading table `data` is queued on `stream` (lets the table be
// retired later without a device-wide synchronisation).
int step_table_used(DeviceCache& dc, const float* data, cudaStream_t stream);

// Axis-pass launchers, one instantiation per label width (edt_passes.cuh).
template <int Bytes>
int launch_first(const void* labels, float* f, int64_t nlines, int64_t sx, float w, int border, int flags,
                 DeviceCache& dc, cudaStream_t stream);
template <int Bytes>
int launch_later(const void* labels, float* f, const LineGeom& g0, float w, int border_lo, int border_hi,
                 int flags, DeviceCache& dc, cudaStream_t stream, bool pdl, double fmax);

}  // namespace host
}  // namespace edtb200
