// edt_capi.cu -- host side of the C ABI declared in include/edt_b200.h.
//
// Plays the role of the reference's volume drivers (pyedt::_edt3dsq / _edt2dsq,
// src/edt.hpp:411-484, 632-678): it owns the pass order X -> Y -> Z over one float32
// volume that is transformed in place, but the "thread pool" is the CUDA grid and the
// passes are stream-ordered kernel launches.  No CPU fallback exists in this file.
#include "edt_host.h"
#include "edt_voxel_graph.cuh"
#include "edt_each.cuh"
#include "edt_slab.cuh"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

namespace edtb200 {
namespace host {

thread_local char g_error[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
  return code;
}

EncodeTiledFn tensor_map_encoder() {
  static std::once_flag once;
  static EncodeTiledFn encode = nullptr;
  std::call_once(once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      encode = reinterpret_cast<EncodeTiledFn>(fn);
    else
      cudaGetLastError();
  });
  return encode;
}

cudaError_t scratch_alloc(DeviceCache& dc, void** p, size_t bytes, cudaStream_t stream) {
  if (dc.pool) return cudaMallocFromPoolAsync(p, bytes, dc.pool, stream);
  return cudaMallocAsync(p, bytes, stream);
}

// Device table T[0..count) for weight w, cached per device.  Built once on `stream`; other
// streams wait on the build event, so no host synchronisation and no per-call allocation.
// When all slots are taken the least recently used table is retired: the retiring stream waits
// for the last kernel of every stream that used the table (one event per user stream) and the
// buffer is freed in stream order -- no device-wide synchronisation.
int step_table(DeviceCache& dc, float w, int count, cudaStream_t stream, const float** out) {
  std::lock_guard<std::mutex> guard(dc.lock);
  uint32_t wbits;
  memcpy(&wbits, &w, sizeof(wbits));
  DeviceCache::Table* hit = nullptr;
  DeviceCache::Table* victim = &dc.tables[0];
  for (auto& t : dc.tables) {
    if (t.data && t.wbits == wbits && t.count >= count) { hit = &t; break; }
    if (t.stamp < victim->stamp) victim = &t;
  }
  if (!hit) {
    DeviceCache::Table& t = *victim;
    if (t.data) {
      if (t.many_users) CUDA_TRY(cudaDeviceSynchronize());    // more user streams than tracked: rare
      for (int u = 0; u < DeviceCache::Table::kUsers; ++u)
        if (t.user_set[u]) CUDA_TRY(cudaStreamWaitEvent(stream, t.used[u], 0));
      if (t.ready) CUDA_TRY(cudaStreamWaitEvent(stream, t.ready, 0));
      CUDA_TRY(cudaFreeAsync(t.data, stream));
      t.data = nullptr;
      for (int u = 0; u < DeviceCache::Table::kUsers; ++u) t.user_set[u] = false;
      t.many_users = false;
    }
    const int cap = count < 4096 ? 4096 : count;
    CUDA_TRY(scratch_alloc(dc, reinterpret_cast<void**>(&t.data), sizeof(float) * (size_t)cap, stream));
    if (!t.ready) CUDA_TRY(cudaEventCreateWithFlags(&t.ready, cudaEventDisableTiming));
    step_table_kernel<<<1, 32, 0, stream>>>(w, cap, t.data);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(t.ready, stream));
    t.count = cap; t.wbits = wbits; t.built_on = stream;
    hit = &t;
  } else if (hit->built_on != stream) {
    CUDA_TRY(cudaStreamWaitEvent(stream, hit->ready, 0));
  }
  hit->stamp = ++dc.table_clock;
  *out = hit->data;
  return 0;
}

// Called after the kernel that reads table `data` has been queued on `stream`.
int step_table_used(DeviceCache& dc, const float* data, cudaStream_t stream) {
  std::lock_guard<std::mutex> guard(dc.lock);
  for (auto& t : dc.tables) {
    if (t.data != data) continue;
    int slot = -1;
    for (int u = 0; u < DeviceCache::Table::kUsers; ++u)
      if (t.user_set[u] && t.user[u] == stream) { slot = u; break; }
    if (slot < 0)
      for (int u = 0; u < DeviceCache::Table::kUsers; ++u)
        if (!t.user_set[u]) { slot = u; break; }
    if (slot < 0) { t.many_users = true; return 0; }
    if (!t.used[slot]) CUDA_TRY(cudaEventCreateWithFlags(&t.used[slot], cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(t.used[slot], stream));
    t.user[slot] = stream; t.user_set[slot] = true;
    return 0;
  }
  return 0;
}

}  // namespace host
}  // namespace edtb200

namespace {

using namespace edtb200::host;

constexpr int kMaxDevices = 64;
DeviceCache g_cache[kMaxDevices];

// ---- host <-> device staging for pageable host memory --------------------------------
// numpy arrays are pageable: a plain cudaMemcpy of 512 MiB then runs at a fraction of the PCIe
// rate (the driver stages it through small internal buffers, and a freshly allocated output
// array is also page-faulted in by that single thread).  Pinned callers are copied directly;
// pageable ones go through three 32 MiB pinned buffers that a few host threads fill / drain in
// parallel while the DMA engine moves the previous chunk.
class CopyPool {
 public:
  explicit CopyPool(int n) : n_(n) {
    for (int i = 0; i < n_; ++i) threads_.emplace_back([this, i] { loop(i); });
  }
  ~CopyPool() {
    { std::lock_guard<std::mutex> l(m_); stop_ = true; ++epoch_; }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
  }
  int size() const { return n_; }
  // run fn(i) for i in [0, n) on the pool and wait
  void run(const std::function<void(int)>& fn) {
    std::unique_lock<std::mutex> l(m_);
    fn_ = &fn; pending_ = n_; ++epoch_;
    cv_.notify_all();
    done_.wait(l, [this] { return pending_ == 0; });
    fn_ = nullptr;
  }
 private:
  void loop(int i) {
    unsigned long seen = 0;
    for (;;) {
      const std::function<void(int)>* fn;
      {
        std::unique_lock<std::mutex> l(m_);
        cv_.wait(l, [&] { return epoch_ != seen; });
        seen = epoch_;
        if (stop_) return;
        fn = fn_;
      }
      (*fn)(i);
      {
        std::lock_guard<std::mutex> l(m_);
        if (--pending_ == 0) done_.notify_all();
      }
    }
  }
  int n_;
  std::vector<std::thread> threads_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<void(int)>* fn_ = nullptr;
  int pending_ = 0;
  unsigned long epoch_ = 0;
  bool stop_ = false;
};

// Per device, two pools and two sets of staging buffers: [0] for copies towards the device, [1]
// for copies back, so that a batch (edtb200_transform_batch) can drive both directions at once
// from two host threads, and calls on different devices never share a pool.  Created on first use
// (under g_init); used only by the holder of the device's host_call lock and its batch helper.
std::mutex g_init;
CopyPool* g_pools[2][kMaxDevices] = {};

void parallel_memcpy(void* dst, const void* src, size_t bytes, int dir, int device) {
  CopyPool*& g_pool = g_pools[dir][device];
  if (!g_pool) {
    std::lock_guard<std::mutex> guard(g_init);
    unsigned hw = std::thread::hardware_concurrency();
    // measured on the B200 host (2 x 64 threads), 512 MiB each way: 8 threads 40 ms, 16 threads
    // 31 ms, 32 threads 38 ms per numpy-to-numpy call; populating the fresh output array's pages
    // from helper threads during the upload was tried and only made it slower (44-68 ms)
    int n = hw >= 48 ? 24 : (hw >= 32 ? 16 : (hw >= 16 ? 8 : (hw >= 4 ? 4 : 1)));     // r02 sweep: 24 threads 22-25 ms, 16: 25-27, 32: 27
    if (const char* e = getenv("EDTB200_COPY_THREADS")) n = std::max(1, std::min(64, atoi(e)));
    g_pool = new CopyPool(n);
  }
  const int n = g_pool->size();
  const size_t slice = ((bytes + n - 1) / n + 4095) & ~size_t(4095);
  g_pool->run([&](int i) {
    const size_t off = slice * (size_t)i;
    if (off < bytes) memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off,
                            bytes - off < slice ? bytes - off : slice);
  });
}

// size of one staging buffer (EDTB200_STAGE_MB, 4..256, default 32) and how many rotate
const size_t kStageBytes = [] {
  size_t mb = 32;
  if (const char* e = getenv("EDTB200_STAGE_MB")) mb = (size_t)std::max(4, std::min(256, atoi(e)));
  return mb << 20;
}();
constexpr int kStages = 3;
struct StageBuffers {
  void* buf[kStages] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev[kStages] = {nullptr, nullptr, nullptr};
};
StageBuffers g_stage[2][kMaxDevices];

bool host_pointer_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

int ensure_stage(int device, int dir) {
  StageBuffers& sb = g_stage[dir][device];
  for (int i = 0; i < kStages; ++i) {
    if (!sb.buf[i]) CUDA_TRY(cudaHostAlloc(&sb.buf[i], kStageBytes, cudaHostAllocDefault));
    if (!sb.ev[i]) CUDA_TRY(cudaEventCreateWithFlags(&sb.ev[i], cudaEventDisableTiming));
  }
  return 0;
}

// host (pageable or pinned) -> device, stream-ordered; returns after the last chunk is queued
int upload(void* dst_dev, const void* src_host, size_t bytes, int device, cudaStream_t stream) {
  if (bytes < (size_t(4) << 20) || host_pointer_is_pinned(src_host)) {
    CUDA_TRY(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, stream));
    return 0;
  }
  int rc = ensure_stage(device, 0);
  if (rc) return rc;
  StageBuffers& sb = g_stage[0][device];
  size_t off = 0;
  for (int k = 0; off < bytes; ++k) {
    const int b = k % kStages;
    const size_t n = bytes - off < kStageBytes ? bytes - off : kStageBytes;
    // the DMA out of this buffer must have finished -- also the one queued by an EARLIER upload:
    // inside a batch the previous volume's copies may still be waiting in the stream
    CUDA_TRY(cudaEventSynchronize(sb.ev[b]));
    parallel_memcpy(sb.buf[b], static_cast<const char*>(src_host) + off, n, 0, device);
    CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(dst_dev) + off, sb.buf[b], n, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaEventRecord(sb.ev[b], stream));
    off += n;
  }
  return 0;
}

// device -> host (pageable or pinned); complete on return for the pageable case
int download(void* dst_host, const void* src_dev, size_t bytes, int device, cudaStream_t stream) {
  if (bytes < (size_t(4) << 20) || host_pointer_is_pinned(dst_host)) {
    CUDA_TRY(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, stream));
    return 0;
  }
  int rc = ensure_stage(device, 1);
  if (rc) return rc;
  StageBuffers& sb = g_stage[1][device];
  size_t off = 0, prev_off = 0, prev_n = 0;
  int prev_b = -1;
  for (int k = 0; off < bytes || prev_b >= 0; ++k) {
    int b = -1;
    size_t n = 0;
    if (off < bytes) {
      b = k % kStages;
      n = bytes - off < kStageBytes ? bytes - off : kStageBytes;
      CUDA_TRY(cudaMemcpyAsync(sb.buf[b], static_cast<const char*>(src_dev) + off, n, cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaEventRecord(sb.ev[b], stream));
    }
    if (prev_b >= 0) {                                             // drain the chunk queued one step earlier
      CUDA_TRY(cudaEventSynchronize(sb.ev[prev_b]));
      parallel_memcpy(static_cast<char*>(dst_host) + prev_off, sb.buf[prev_b], prev_n, 1, device);
    }
    prev_b = b; prev_off = off; prev_n = n;
    off += n;
  }
  return 0;
}

// Restores the calling thread's current CUDA device when an entry point returns (callers such as
// PyTorch rely on "their" current device staying put).
struct DeviceGuard {
  int saved = -1;
  DeviceGuard() { if (cudaGetDevice(&saved) != cudaSuccess) { cudaGetLastError(); saved = -1; } }
  ~DeviceGuard() { if (saved >= 0) cudaSetDevice(saved); }
};

int probe(int device, DeviceCache** out) {
  if (device < 0 || device >= kMaxDevices) return fail(EDTB200_EINVAL, "bad device %d", device);
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(EDTB200_ECUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device >= count) return fail(EDTB200_EINVAL, "device %d out of range (%d visible)", device, count);
  DeviceCache& dc = g_cache[device];
  CUDA_TRY(cudaSetDevice(device));
  std::lock_guard<std::mutex> guard(dc.lock);
  if (!dc.probed) {
    CUDA_TRY(cudaDeviceGetAttribute(&dc.sm_count, cudaDevAttrMultiProcessorCount, device));
    CUDA_TRY(cudaDeviceGetAttribute(&dc.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    // Stream-ordered scratch (voxel-graph grids, long-line temporaries, step tables) comes from a
    // PRIVATE pool: the process-wide default pool -- which the host application (PyTorch, CuPy)
    // may share -- keeps its own settings.  The pool keeps up to EDTB200_POOL_KEEP_MB (default
    // 1024) between calls so that repeated transforms do not go back to the driver;
    // edtb200_release() trims it to nothing.
    cudaMemPoolProps props;
    memset(&props, 0, sizeof(props));
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if (cudaMemPoolCreate(&dc.pool, &props) == cudaSuccess) {
      unsigned long long keep = 1024ull << 20;
      if (const char* env = getenv("EDTB200_POOL_KEEP_MB")) keep = strtoull(env, nullptr, 10) << 20;
      cudaMemPoolSetAttribute(dc.pool, cudaMemPoolAttrReleaseThreshold, &keep);
    } else {
      dc.pool = nullptr;                 // fall back to the default pool, settings untouched
    }
    cudaGetLastError();
    // run statistic of the first-axis pass: two device counters and two mapped host words
    void* stat = nullptr;
    void* host = nullptr;
    if (cudaMalloc(&stat, 64) == cudaSuccess && cudaMemset(stat, 0, 64) == cudaSuccess &&
        cudaHostAlloc(&host, 64, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
      memset(host, 0, 64);
      void* host_dev = nullptr;
      if (cudaHostGetDevicePointer(&host_dev, host, 0) == cudaSuccess) {
        dc.stat_counter = static_cast<unsigned long long*>(stat);
        dc.stat_ticket = reinterpret_cast<unsigned int*>(static_cast<char*>(stat) + 16);
        dc.stat_publish_host = static_cast<volatile unsigned long long*>(host);
        dc.stat_publish_dev = static_cast<unsigned long long*>(host_dev);
      }
    }
    cudaGetLastError();
    dc.probed = true;
  }
  *out = &dc;
  return 0;
}

int check_dims(int label_bytes, int ndim, int64_t& sx, int64_t& sy, int64_t& sz) {
  if (!(label_bytes == 1 || label_bytes == 2 || label_bytes == 4 || label_bytes == 8))
    return fail(EDTB200_EINVAL, "label_bytes must be 1, 2, 4 or 8 (got %d)", label_bytes);
  if (ndim < 1 || ndim > 3) return fail(EDTB200_EINVAL, "ndim must be 1, 2 or 3 (got %d)", ndim);
  if (ndim < 3) sz = 1;
  if (ndim < 2) sy = 1;
  if (sx < 0 || sy < 0 || sz < 0) return fail(EDTB200_EINVAL, "negative size");
  const int64_t lim = (int64_t)1 << 30;
  if (sx > lim || sy > lim || sz > lim) return fail(EDTB200_ELIMIT, "axis longer than 2^30");
  return 0;
}

template <int B>
struct LabelWidth {
  static constexpr int Bytes = B;
  using T = typename edtb200::LabelOf<B>::type;
};

// f(LabelWidth<label_bytes>()): the label width as a compile-time constant (check_dims has
// accepted it: 1, 2, 4 or 8).
template <class F>
auto with_label_width(int label_bytes, F&& f) {
  switch (label_bytes) {
    case 1: return f(LabelWidth<1>());
    case 2: return f(LabelWidth<2>());
    case 4: return f(LabelWidth<4>());
    default: return f(LabelWidth<8>());
  }
}

// Kernel flags of the pass that ends a transform: square root, and the sign of sdf.
int epilogue_flags(int flags) {
  return ((flags & EDTB200_SQRT) ? edtb200::kSqrt : 0) | ((flags & EDTB200_SIGNED) ? edtb200::kNegate : 0);
}

// Kernel flag of sdf's first pass: the background (label 0) is a label like any other.
int zero_label_flags(int flags) { return (flags & EDTB200_SIGNED) ? edtb200::kZeroLabel : 0; }

// Largest finite value the passes along axes of lengths n[0..k) with weights w[0..k) can have
// produced, if all their squared weights (the float products the kernels use) are integers and
// the distances stay exact in float32; else -1.  (An X-pass value is fl32(a_k^2) with a_k = k*w
// exact below 2^24; a later pass adds w2 * d^2 to an earlier value.)
double integer_bound(const float* w, const int64_t* n, int k) {
  double bound = 0.0;
  for (int i = 0; i < k; ++i) {
    const float w2 = w[i] * w[i];
    if (!(w2 == floorf(w2)) || w2 < 1.0f) return -1.0;
    if (i == 0 && !((double)w[0] == floor((double)w[0]) && (double)w[0] * (double)n[0] < 16777216.0)) return -1.0;
    bound += (double)w2 * (double)n[i] * (double)n[i];
  }
  return bound < 2147483000.0 ? bound : -1.0;
}

// {outer_count, outer_stride, inner_count, line_stride, n, tiles_per_outer} of the Y / Z pass
edtb200::LineGeom geom_for_axis(int axis, int64_t sx, int64_t sy, int64_t sz) {
  if (axis == 1) return {sz, sx * sy, sx, sx, (int)sy, 0};
  return {1, 0, sx * sy, sx * sy, (int)sz, 0};
}

int first_pass(int label_bytes, const void* labels, float* f, int64_t nlines, int64_t sx, float wx, int border,
               int kflags, DeviceCache& dc, cudaStream_t s) {
  return with_label_width(label_bytes, [&](auto lw) {
    return launch_first<decltype(lw)::Bytes>(labels, f, nlines, sx, wx, border, kflags, dc, s);
  });
}

// The Y (axis 1) or Z (axis 2) pass of a volume of sx x sy x sz voxels with weights w[0..2], after
// the passes along the earlier axes.  `part` is the extent the call covers across its lines -- z
// for Y, y for Z: sz / sy, or one device's share when the volume is split; the integer-hull bound
// is that of the whole volume.
int later_pass(int axis, int label_bytes, const void* labels, float* f, int64_t sx, int64_t sy, int64_t sz,
               int64_t part, const float* w, int border_lo, int border_hi, int kflags, bool pdl, DeviceCache& dc,
               cudaStream_t s) {
  const int64_t n[2] = {sx, sy};
  const edtb200::LineGeom g = axis == 1 ? geom_for_axis(1, sx, sy, part) : geom_for_axis(2, sx, part, sz);
  return with_label_width(label_bytes, [&](auto lw) {
    return launch_later<decltype(lw)::Bytes>(labels, f, g, w[axis], border_lo, border_hi, kflags, dc, s, pdl,
                                             integer_bound(w, n, axis));
  });
}

// Device buffer `p` of at least `need` bytes (`have` now), reallocated when too small.
template <class T>
cudaError_t grow(T*& p, size_t& have, size_t need) {
  if (have >= need) return cudaSuccess;
  if (p) cudaFree(p);
  p = nullptr; have = 0;
  const cudaError_t e = cudaMalloc(&p, need);
  if (e == cudaSuccess) have = need;
  return e;
}

// Creates the cached non-blocking stream `s` of a device on first use.
cudaError_t ensure_stream(cudaStream_t& s) {
  return s ? cudaSuccess : cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
}

// Optional per-pass timing for bench.py: with profiling on, every transform of this thread records
// four CUDA events (before / between / after its axis passes) into a ring, so a timed loop can be
// analysed afterwards without any synchronisation inside it (edtb200_profile_passes /
// edtb200_pass_ms).
constexpr int kProfileRing = 256;
thread_local bool g_profile = false;
thread_local cudaEvent_t g_pass_events[kProfileRing][4];
thread_local bool g_pass_events_init = false;
thread_local int g_pass_marks[kProfileRing];       // highest mark index recorded in the slot
thread_local long g_pass_seq = 0;                  // transforms profiled so far

void mark_pass(int idx, cudaStream_t stream) {
  if (!g_profile) return;
  if (!g_pass_events_init) {
    for (auto& slot : g_pass_events) for (auto& e : slot) e = nullptr;
    g_pass_events_init = true;
  }
  if (idx == 0) ++g_pass_seq;
  const int slot = (int)((g_pass_seq - 1) % kProfileRing);
  cudaEvent_t& e = g_pass_events[slot][idx];
  if (!e && cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); return; }
  cudaEventRecord(e, stream);
  g_pass_marks[slot] = idx;
}

// NVTX ranges edt.x / edt.y / edt.z / edt.halo.* (SURVEY.md section 5) around the launches, so
// that an Nsight Systems timeline names the passes.  libnvToolsExt is looked up at run time
// (dlopen), so it is not a dependency; without it the calls do nothing.
typedef int (*NvtxPushFn)(const char*);
typedef int (*NvtxPopFn)(void);
NvtxPushFn g_nvtx_push = nullptr;
NvtxPopFn g_nvtx_pop = nullptr;
std::once_flag g_nvtx_once;

void nvtx_init() {
  std::call_once(g_nvtx_once, [] {
    if (getenv("EDTB200_NO_NVTX")) return;
    const char* names[] = {"libnvToolsExt.so.1", "libnvToolsExt.so", nullptr};
    for (int i = 0; names[i]; ++i) {
      void* h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
      if (!h) continue;
      g_nvtx_push = reinterpret_cast<NvtxPushFn>(dlsym(h, "nvtxRangePushA"));
      g_nvtx_pop = reinterpret_cast<NvtxPopFn>(dlsym(h, "nvtxRangePop"));
      if (g_nvtx_push && g_nvtx_pop) return;
      g_nvtx_push = nullptr; g_nvtx_pop = nullptr;
    }
  });
}
void nvtx_push(const char* name) { nvtx_init(); if (g_nvtx_push) g_nvtx_push(name); }
void nvtx_pop() { if (g_nvtx_pop) g_nvtx_pop(); }

// All passes of one transform on device-resident buffers.
int run_passes(const void* labels, int label_bytes, int ndim, int64_t sx, int64_t sy, int64_t sz,
               float wx, float wy, float wz, int border, int flags, float* f,
               DeviceCache& dc, cudaStream_t stream) {
  // sqrt / sign are applied by whichever pass is the last one; background-as-label (sdf)
  // changes the first pass only -- later passes treat every run alike.
  const int epilogue = epilogue_flags(flags);
  const float w[3] = {wx, wy, wz};
  // The later passes are launched with programmatic stream serialization: the kernel before them
  // in the stream is our own previous pass, which never writes the labels, so their label staging
  // (before griddepcontrol.wait) may overlap its tail.  The per-axis entry points do not do this:
  // there the previous kernel is the caller's and may be the one producing the labels.
  // (A one-byte neighbour-code plane written by the first pass, so that the later passes need not
  // re-read wide labels, was measured in round 1 and dropped: Y 0.261 -> 0.244, Z 0.280 -> 0.250 ms
  // but X 0.180 -> 0.350 ms at 512^3 uint32.)
  int rc = 0;
  // EDT_B200_VERBOSE=1: per-pass device times of every transform on stderr (SURVEY.md section 5).
  // The dump needs the passes to have finished, so a verbose transform synchronises its stream.
  static const bool verbose = getenv("EDT_B200_VERBOSE") != nullptr && atoi(getenv("EDT_B200_VERBOSE")) != 0;
  const bool profile_was = g_profile;
  if (verbose) g_profile = true;
  mark_pass(0, stream);
  nvtx_push("edt.x");
  rc = first_pass(label_bytes, labels, f, sy * sz, sx, wx, border,
                  zero_label_flags(flags) | (ndim == 1 ? epilogue : 0), dc, stream);
  nvtx_pop();
  mark_pass(1, stream);
  if (!rc && ndim >= 2) {
    nvtx_push("edt.y");
    rc = later_pass(1, label_bytes, labels, f, sx, sy, sz, sz, w, border, border, ndim == 2 ? epilogue : 0,
                    /*pdl=*/true, dc, stream);
    nvtx_pop();
    mark_pass(2, stream);
  }
  if (!rc && ndim >= 3) {
    nvtx_push("edt.z");
    rc = later_pass(2, label_bytes, labels, f, sx, sy, sz, sy, w, border, border, epilogue, /*pdl=*/true, dc,
                    stream);
    nvtx_pop();
    mark_pass(3, stream);
  }
  if (verbose) {
    g_profile = profile_was;
    float ms[3] = {0.0f, 0.0f, 0.0f};
    if (!rc && edtb200_pass_ms(0, ms) == 0) {
      const double nvox = (double)sx * (double)sy * (double)sz;
      const double total = ms[0] + ms[1] + ms[2];
      fprintf(stderr, "[edt_b200] %lldx%lldx%lld L=%d  x %.3f ms  y %.3f ms  z %.3f ms  total %.3f ms  "
                      "%.0f Mvox/s  %.0f GB/s algorithmic\n",
              (long long)sx, (long long)sy, (long long)sz, label_bytes, ms[0], ms[1], ms[2], total,
              total > 0 ? nvox / total / 1e3 : 0.0,
              total > 0 ? nvox * (3.0 * label_bytes + 20.0) / total / 1e6 : 0.0);
    }
  }
  return rc;
}


}  // namespace

extern "C" {

int edtb200_version(void) { return EDTB200_VERSION; }

const char* edtb200_last_error(void) { return g_error; }

int edtb200_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
  return count;
}

int edtb200_transform(const void* labels, int label_bytes, int ndim, int64_t sx, int64_t sy, int64_t sz,
                      float wx, float wy, float wz, int black_border, int flags, float* out,
                      int device, void* stream_v) {
  int rc = check_dims(label_bytes, ndim, sx, sy, sz);
  if (rc) return rc;
  const int64_t total = sx * sy * sz;
  if (total == 0) return 0;
  if (!labels || !out) return fail(EDTB200_EINVAL, "null pointer");

  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;

  const bool lab_dev = flags & EDTB200_LABELS_ON_DEVICE;
  const bool out_dev = flags & EDTB200_OUT_ON_DEVICE;
  const int border = black_border != 0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);

  // device-resident: asynchronous on the caller's stream, no library-wide or per-device lock held
  if (lab_dev && out_dev)
    return run_passes(labels, label_bytes, ndim, sx, sy, sz, wx, wy, wz, border, flags, out, *dc, stream);

  // host memory involved: stage through this device's cached buffers, synchronous on return.
  // Calls on other devices proceed concurrently (per-device lock).
  std::lock_guard<std::mutex> host_call(dc->host_call);
  if (!stream && !lab_dev && !out_dev) {
    // pure host call: a private non-blocking stream.  With one side on the device and no stream
    // given, the legacy default stream (NULL) is kept: it is ordered after the work the caller
    // queued on the default / blocking streams that produced that buffer.
    CUDA_TRY(ensure_stream(dc->stream));
    stream = dc->stream;
  }
  const size_t lab_bytes = (size_t)total * (size_t)label_bytes;
  const size_t out_bytes = (size_t)total * sizeof(float);
  const void* d_labels = labels;
  float* d_out = out;
  if (!lab_dev) {
    CUDA_TRY(grow(dc->labels, dc->labels_bytes, lab_bytes));
    rc = upload(dc->labels, labels, lab_bytes, device, stream);
    if (rc) return rc;
    d_labels = dc->labels;
  }
  if (!out_dev) {
    CUDA_TRY(grow(dc->dist, dc->dist_bytes, out_bytes));
    d_out = dc->dist;
  }
  rc = run_passes(d_labels, label_bytes, ndim, sx, sy, sz, wx, wy, wz, border, flags, d_out, *dc, stream);
  if (rc) return rc;
  if (!out_dev) {
    rc = download(out, d_out, out_bytes, device, stream);
    if (rc) return rc;
  }
  CUDA_TRY(cudaStreamSynchronize(stream));
  return 0;
}

int edtb200_transform_batch(const void* const* labels, float* const* outs, int count, int label_bytes, int ndim,
                            int64_t sx, int64_t sy, int64_t sz, float wx, float wy, float wz,
                            int black_border, int flags, int device) {
  if (count < 0) return fail(EDTB200_EINVAL, "negative count");
  if (flags & (EDTB200_LABELS_ON_DEVICE | EDTB200_OUT_ON_DEVICE))
    return fail(EDTB200_EINVAL, "edtb200_transform_batch pipelines HOST buffers; device-resident volumes are "
                                "already asynchronous through edtb200_transform");
  int rc = check_dims(label_bytes, ndim, sx, sy, sz);
  if (rc) return rc;
  const int64_t total = sx * sy * sz;
  if (total == 0 || count == 0) return 0;
  if (!labels || !outs) return fail(EDTB200_EINVAL, "null pointer");
  for (int k = 0; k < count; ++k)
    if (!labels[k] || !outs[k]) return fail(EDTB200_EINVAL, "null pointer in volume %d", k);

  DeviceGuard restore_device;
  DeviceCache* dcp = nullptr;
  rc = probe(device, &dcp);
  if (rc) return rc;
  DeviceCache& dc = *dcp;
  std::lock_guard<std::mutex> host_call(dc.host_call);
  const size_t lab_bytes = (size_t)total * (size_t)label_bytes, out_bytes = (size_t)total * sizeof(float);
  CUDA_TRY(grow(dc.labels, dc.labels_bytes, lab_bytes));
  CUDA_TRY(grow(dc.dist, dc.dist_bytes, out_bytes));
  if (count > 1) {
    CUDA_TRY(grow(dc.labels2, dc.labels2_bytes, lab_bytes));
    CUDA_TRY(grow(dc.dist2, dc.dist2_bytes, out_bytes));
  }
  CUDA_TRY(ensure_stream(dc.stream));
  CUDA_TRY(ensure_stream(dc.stream_up));
  CUDA_TRY(ensure_stream(dc.stream_down));
  for (int i = 0; i < 2; ++i) {
    if (!dc.ev_up[i]) CUDA_TRY(cudaEventCreateWithFlags(&dc.ev_up[i], cudaEventDisableTiming));
    if (!dc.ev_comp[i]) CUDA_TRY(cudaEventCreateWithFlags(&dc.ev_comp[i], cudaEventDisableTiming));
    if (!dc.ev_down[i]) CUDA_TRY(cudaEventCreateWithFlags(&dc.ev_down[i], cudaEventDisableTiming));
  }
  void* d_labels[2] = {dc.labels, dc.labels2};
  float* d_dist[2] = {dc.dist, dc.dist2};
  const int border = black_border != 0;

  // Volume k uses slot k % 2.  Three streams: uploads (fed by a helper thread, so that pageable
  // buffers can be staged in both directions at once), the passes, downloads (this thread).
  //   upload k    waits for the passes of k-2 (they read the slot's labels)
  //   passes k    wait for upload k and for download k-2 (it reads the slot's distances)
  //   download k  waits for the passes of k
  // Host-side counters make sure an event has been RECORDED before someone waits on it.
  std::mutex m;
  std::condition_variable cv;
  int uploads_queued = 0, passes_queued = 0, failed = 0;
  char upload_error[sizeof(g_error)] = "";
  std::thread uploader([&] {
    cudaSetDevice(device);
    for (int k = 0; k < count; ++k) {
      const int slot = k & 1;
      int urc = 0;
      if (k >= 2) {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { return passes_queued >= k - 1 || failed; });
        if (failed) return;
        if (cudaStreamWaitEvent(dc.stream_up, dc.ev_comp[slot], 0) != cudaSuccess) urc = EDTB200_ECUDA;
      }
      if (!urc) urc = upload(d_labels[slot], labels[k], lab_bytes, device, dc.stream_up);
      if (!urc && cudaEventRecord(dc.ev_up[slot], dc.stream_up) != cudaSuccess) urc = EDTB200_ECUDA;
      std::lock_guard<std::mutex> l(m);
      if (urc) {
        failed = urc;
        snprintf(upload_error, sizeof(upload_error), "upload of volume %d failed: %.400s", k,
                 urc == EDTB200_ECUDA ? cudaGetErrorString(cudaGetLastError()) : g_error);
      } else {
        uploads_queued = k + 1;
      }
      cv.notify_all();
      if (urc) return;
    }
  });
  auto bail = [&](int code) {
    { std::lock_guard<std::mutex> l(m); if (!failed) failed = code; }
    cv.notify_all();
    uploader.join();
    cudaStreamSynchronize(dc.stream_up); cudaStreamSynchronize(dc.stream); cudaStreamSynchronize(dc.stream_down);
    return code;
  };
  #define BATCH_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { \
      fail(EDTB200_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_)); return bail(EDTB200_ECUDA); } } while (0)
  for (int k = 0; k < count; ++k) {
    const int slot = k & 1;
    {
      std::unique_lock<std::mutex> l(m);
      cv.wait(l, [&] { return uploads_queued >= k + 1 || failed; });
      if (failed) { l.unlock(); uploader.join(); cudaDeviceSynchronize(); return fail(failed, "%s", upload_error); }
    }
    BATCH_TRY(cudaStreamWaitEvent(dc.stream, dc.ev_up[slot], 0));
    if (k >= 2) BATCH_TRY(cudaStreamWaitEvent(dc.stream, dc.ev_down[slot], 0));
    rc = run_passes(d_labels[slot], label_bytes, ndim, sx, sy, sz, wx, wy, wz, border, flags, d_dist[slot], dc,
                    dc.stream);
    if (rc) return bail(rc);
    BATCH_TRY(cudaEventRecord(dc.ev_comp[slot], dc.stream));
    { std::lock_guard<std::mutex> l(m); passes_queued = k + 1; }
    cv.notify_all();
    BATCH_TRY(cudaStreamWaitEvent(dc.stream_down, dc.ev_comp[slot], 0));
    rc = download(outs[k], d_dist[slot], out_bytes, device, dc.stream_down);
    if (rc) return bail(rc);
    BATCH_TRY(cudaEventRecord(dc.ev_down[slot], dc.stream_down));
  }
  #undef BATCH_TRY
  uploader.join();
  CUDA_TRY(cudaStreamSynchronize(dc.stream_down));
  return 0;
}

int edtb200_transform_voxel_graph(const void* labels, int label_bytes, const unsigned char* graph, int ndim,
                                  int64_t sx, int64_t sy, int64_t sz, float wx, float wy, float wz,
                                  int black_border, int flags, float* out, int device, void* stream_v) {
  using namespace edtb200;
  if (ndim != 2 && ndim != 3)
    return fail(EDTB200_EINVAL, "a voxel graph needs a 2-D or 3-D volume (got ndim %d)", ndim);
  if (flags & EDTB200_SIGNED)
    return fail(EDTB200_EINVAL, "EDTB200_SIGNED is not defined with a voxel graph: subtract two transforms");
  if ((flags & EDTB200_LABELS_FLOAT) && label_bytes != 4 && label_bytes != 8)
    return fail(EDTB200_EINVAL, "EDTB200_LABELS_FLOAT needs 4- or 8-byte labels");
  int rc = check_dims(label_bytes, ndim, sx, sy, sz);
  if (rc) return rc;
  const int64_t total = sx * sy * sz;
  if (total == 0) return 0;
  if (!labels || !graph || !out) return fail(EDTB200_EINVAL, "null pointer");
  int64_t sx2 = 2 * sx, sy2 = 2 * sy, sz2 = ndim == 3 ? 2 * sz : 1;
  rc = check_dims(1, ndim, sx2, sy2, sz2);
  if (rc) return rc;
  const int64_t total2 = sx2 * sy2 * sz2;

  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  const bool in_dev = flags & EDTB200_LABELS_ON_DEVICE;
  const bool out_dev = flags & EDTB200_OUT_ON_DEVICE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  std::unique_lock<std::mutex> host_call(dc->host_call, std::defer_lock);
  if (!(in_dev && out_dev)) host_call.lock();          // staging buffers and the private stream
  if (!stream && !in_dev && !out_dev) {
    CUDA_TRY(ensure_stream(dc->stream));
    stream = dc->stream;
  }

  // stream-ordered scratch: the inputs when they come from the host, the doubled byte mask, the
  // doubled distance volume, and the result when it goes back to the host
  void *d_labels = nullptr, *d_graph = nullptr, *d_cells = nullptr, *d_doubled = nullptr, *d_result = nullptr;
  auto release = [&]() {
    void* all[] = {d_labels, d_graph, d_cells, d_doubled, d_result};
    for (void* p : all) if (p) cudaFreeAsync(p, stream);
  };
  #define VG_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { release(); \
      return fail(e_ == cudaErrorMemoryAllocation ? EDTB200_ENOMEM : EDTB200_ECUDA, "%s: %s", #expr, \
                  cudaGetErrorString(e_)); } } while (0)
  const void* lab = labels;
  const uint8_t* gr = graph;
  if (!in_dev) {
    VG_TRY(scratch_alloc(*dc, &d_labels, (size_t)total * label_bytes, stream));
    VG_TRY(scratch_alloc(*dc, &d_graph, (size_t)total, stream));
    rc = upload(d_labels, labels, (size_t)total * label_bytes, device, stream);
    if (!rc) rc = upload(d_graph, graph, (size_t)total, device, stream);
    if (rc) { release(); return rc; }
    lab = d_labels;
    gr = static_cast<const uint8_t*>(d_graph);
  }
  VG_TRY(scratch_alloc(*dc, &d_cells, (size_t)total2, stream));
  VG_TRY(scratch_alloc(*dc, &d_doubled, (size_t)total2 * sizeof(float), stream));
  float* result = out;
  if (!out_dev) {
    VG_TRY(scratch_alloc(*dc, &d_result, (size_t)total * sizeof(float), stream));
    result = static_cast<float*>(d_result);
  }

  const int threads = 256;
  const int blocks = (int)std::min<int64_t>((total + threads - 1) / threads, (int64_t)dc->sm_count * 32);
  const int border = black_border != 0, as_float = (flags & EDTB200_LABELS_FLOAT) ? 1 : 0;
  uint8_t* cells = static_cast<uint8_t*>(d_cells);
  with_label_width(label_bytes, [&](auto lw) {
    voxel_graph_expand_kernel<decltype(lw)::Bytes><<<blocks, threads, 0, stream>>>(lab, gr, cells, sx, sy, sz, ndim,
                                                                                   border, as_float);
  });
  VG_TRY(cudaGetLastError());
  // half the anisotropy (vg:102-107, 199-204); the sqrt is taken by the gather instead
  rc = run_passes(cells, 1, ndim, sx2, sy2, sz2, wx / 2, wy / 2, wz / 2, border, 0,
                  static_cast<float*>(d_doubled), *dc, stream);
  if (rc) { release(); return rc; }
  voxel_graph_gather_kernel<<<blocks, threads, 0, stream>>>(static_cast<const float*>(d_doubled), result, sx, sy, sz,
                                                            (flags & EDTB200_SQRT) ? 1 : 0);
  VG_TRY(cudaGetLastError());
  if (!out_dev) {
    rc = download(out, result, (size_t)total * sizeof(float), device, stream);
    if (rc) { release(); return rc; }
  }
  release();
  if (!(in_dev && out_dev)) VG_TRY(cudaStreamSynchronize(stream));
  #undef VG_TRY
  return 0;
}

int edtb200_pass_first(const void* labels_dev, int label_bytes, int64_t sx, int64_t sy, int64_t sz,
                       float wx, int black_border, int flags, float* f_dev, int device, void* stream) {
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (sx * sy * sz == 0) return 0;
  if (!labels_dev || !f_dev) return fail(EDTB200_EINVAL, "null pointer");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  // EDTB200_SIGNED: background as a label, without the sign
  const int kflags = epilogue_flags(flags & EDTB200_SQRT) | zero_label_flags(flags);
  return first_pass(label_bytes, labels_dev, f_dev, sy * sz, sx, wx, black_border != 0, kflags, *dc,
                    static_cast<cudaStream_t>(stream));
}

int edtb200_pass_later(const void* labels_dev, int label_bytes, int axis, int64_t sx, int64_t sy, int64_t sz,
                       float w, int border_lo, int border_hi, int flags, float* f_dev, int device,
                       void* stream) {
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (axis != 1 && axis != 2) return fail(EDTB200_EINVAL, "axis must be 1 (Y) or 2 (Z)");
  if (sx * sy * sz == 0) return 0;
  if (!labels_dev || !f_dev) return fail(EDTB200_EINVAL, "null pointer");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  const edtb200::LineGeom g = geom_for_axis(axis, sx, sy, sz);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  return with_label_width(label_bytes, [&](auto lw) {      // no integer-hull bound: the caller's f is unknown
    return launch_later<decltype(lw)::Bytes>(labels_dev, f_dev, g, w, border_lo != 0, border_hi != 0,
                                             epilogue_flags(flags), *dc, s, /*pdl=*/false, /*fmax=*/-1.0);
  });
}

int edtb200_slab_face_runs(const void* labels_dev, int label_bytes, int64_t sx, int64_t sy, int64_t sz,
                           int high_face, int halo, int flags, unsigned char* m_dev, int* overflow_dev,
                           int device, void* stream_v) {
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (halo < 1 || halo > 254) return fail(EDTB200_EINVAL, "halo must be in 1..254");
  if (sx * sy * sz == 0) return 0;
  if (!labels_dev || !m_dev || !overflow_dev) return fail(EDTB200_EINVAL, "null pointer");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int64_t plane = sx * sy;
  const unsigned blocks = (unsigned)((plane + 255) / 256);
  const int zl = (flags & EDTB200_SIGNED) ? 1 : 0;
  with_label_width(label_bytes, [&](auto lw) {
    using LW = decltype(lw);
    edtb200::face_runs_kernel<LW::Bytes><<<blocks, 256, 0, stream>>>(
        static_cast<const typename LW::T*>(labels_dev), plane, (int)sz, high_face, halo, zl, m_dev, overflow_dev);
  });
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int edtb200_slab_pack(const void* src_dev, void* dst_dev, int64_t zc, int64_t sy, int64_t row_bytes, int parts,
                      const int64_t* y_start, int unpack, int device, void* stream_v) {
  if (zc < 0 || sy < 0 || row_bytes < 0) return fail(EDTB200_EINVAL, "negative extent");
  if (parts < 1 || parts > 64) return fail(EDTB200_EINVAL, "parts must be in 1..64");
  if (!y_start) return fail(EDTB200_EINVAL, "null pointer");
  edtb200::SlabParts sp;
  sp.n = parts;
  for (int i = 0; i <= parts; ++i) {
    sp.start[i] = y_start[i];
    if ((i == 0 && y_start[i] != 0) || (i > 0 && y_start[i] < y_start[i - 1]))
      return fail(EDTB200_EINVAL, "y_start must rise from 0 to sy");
  }
  if (y_start[parts] != sy) return fail(EDTB200_EINVAL, "y_start must rise from 0 to sy");
  if (zc * sy * row_bytes == 0) return 0;
  if (!src_dev || !dst_dev) return fail(EDTB200_EINVAL, "null pointer");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  int rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int vec16 = (row_bytes % 16 == 0 && reinterpret_cast<uintptr_t>(src_dev) % 16 == 0 &&
                     reinterpret_cast<uintptr_t>(dst_dev) % 16 == 0) ? 1 : 0;
  const int64_t rows = zc * sy;
  const unsigned blocks = (unsigned)std::min<int64_t>(rows, (int64_t)dc->sm_count * 32);
  const unsigned char* a = static_cast<const unsigned char*>(src_dev);
  unsigned char* b = static_cast<unsigned char*>(dst_dev);
  if (unpack) edtb200::slab_pack_kernel<true><<<blocks, 256, 0, stream>>>(a, b, zc, sy, row_bytes, vec16, sp);
  else edtb200::slab_pack_kernel<false><<<blocks, 256, 0, stream>>>(a, b, zc, sy, row_bytes, vec16, sp);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int edtb200_slab_face_fixup(const void* labels_dev, int label_bytes, int64_t sx, int64_t sy, int64_t sz,
                            int high_face, int halo, float wz, int flags, const void* nb_label_dev,
                            const unsigned char* nb_m_dev, const float* nb_f_dev, float* f_dev, int* inexact_dev,
                            int device, void* stream_v) {
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (halo < 1 || halo > 254) return fail(EDTB200_EINVAL, "halo must be in 1..254");
  if (sx * sy * sz == 0) return 0;
  if (!labels_dev || !nb_label_dev || !nb_m_dev || !nb_f_dev || !f_dev) return fail(EDTB200_EINVAL, "null pointer");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int64_t plane = sx * sy;
  const unsigned blocks = (unsigned)((plane + 255) / 256);
  const int kflags = epilogue_flags(flags) | zero_label_flags(flags);
  const float w2 = wz * wz;
  with_label_width(label_bytes, [&](auto lw) {
    using LW = decltype(lw);
    edtb200::face_fixup_kernel<LW::Bytes><<<blocks, 256, 0, stream>>>(
        static_cast<const typename LW::T*>(labels_dev), f_dev, plane, (int)sz, high_face, halo, w2,
        static_cast<const typename LW::T*>(nb_label_dev), nb_m_dev, nb_f_dev, kflags, inexact_dev);
  });
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- one host volume on several GPUs of this process ---------------------------------------
// Z slabs for the X and Y passes, Y slabs (whole z lines) for the Z pass: between the two the
// distances and labels are re-partitioned by peer-to-peer 3-D copies over NVLink, so the result is
// exact for any input with no halo and no verdict -- for a HOST volume the PCIe copies dominate
// anyway and every GPU brings its own link.  One host thread per device; the threads meet at two
// barriers (after the Y passes, after the Z passes), the devices through events.
namespace {

struct MultiBarrier {
  std::mutex m;
  std::condition_variable cv;
  int waiting = 0, generation = 0, parties = 0, failed = 0;
  // returns the failure code agreed by all parties (0 = go on)
  int arrive(int my_rc) {
    std::unique_lock<std::mutex> l(m);
    if (my_rc && !failed) failed = my_rc;
    const int gen = generation;
    if (++waiting == parties) { waiting = 0; ++generation; cv.notify_all(); }
    else cv.wait(l, [&] { return generation != gen; });
    return failed;
  }
};

struct MultiPart {
  int device = 0;
  int64_t z0 = 0, zc = 0, y0 = 0, yc = 0;
  void* lz = nullptr; float* fz = nullptr; void* ly = nullptr; float* fy = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t after_y = nullptr, after_z = nullptr;
  char error[256] = "";
};

cudaError_t copy_box(void* dst, size_t dst_row_bytes, int64_t dst_rows_per_slice, int dst_dev, int64_t dx_bytes,
                     int64_t dy, int64_t dz, const void* src, size_t src_row_bytes, int64_t src_rows_per_slice,
                     int src_dev, int64_t sx_bytes, int64_t sy0, int64_t sz0, size_t width_bytes, int64_t height,
                     int64_t depth, cudaStream_t stream) {
  cudaMemcpy3DPeerParms p;
  memset(&p, 0, sizeof(p));
  p.srcDevice = src_dev;
  p.dstDevice = dst_dev;
  p.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src), src_row_bytes, src_row_bytes, (size_t)src_rows_per_slice);
  p.dstPtr = make_cudaPitchedPtr(dst, dst_row_bytes, dst_row_bytes, (size_t)dst_rows_per_slice);
  p.srcPos = make_cudaPos((size_t)sx_bytes, (size_t)sy0, (size_t)sz0);
  p.dstPos = make_cudaPos((size_t)dx_bytes, (size_t)dy, (size_t)dz);
  p.extent = make_cudaExtent(width_bytes, (size_t)height, (size_t)depth);
  return cudaMemcpy3DPeerAsync(&p, stream);
}

}  // namespace

int edtb200_transform_multi(const void* labels, int label_bytes, int ndim, int64_t sx, int64_t sy, int64_t sz,
                            float wx, float wy, float wz, int black_border, int flags, float* out,
                            const int* devices, int ndevices) {
  if (!devices || ndevices < 1) return fail(EDTB200_EINVAL, "no devices given");
  if (flags & (EDTB200_LABELS_ON_DEVICE | EDTB200_OUT_ON_DEVICE))
    return fail(EDTB200_EINVAL, "edtb200_transform_multi splits a HOST volume over the devices");
  int rc = check_dims(label_bytes, ndim, sx, sy, sz);
  if (rc) return rc;
  if (sx * sy * sz == 0) return 0;
  if (!labels || !out) return fail(EDTB200_EINVAL, "null pointer");
  for (int i = 0; i < ndevices; ++i)
    for (int j = 0; j < i; ++j)
      if (devices[i] == devices[j]) return fail(EDTB200_EINVAL, "device %d listed twice", devices[i]);
  int G = ndevices;
  if (ndim < 3) G = 1;
  if (G > sz) G = (int)sz;
  if (G > sy) G = (int)sy;
  if (G <= 1)
    return edtb200_transform(labels, label_bytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags, out, devices[0],
                             nullptr);

  const int border = black_border != 0;
  const float w[3] = {wx, wy, wz};
  std::vector<MultiPart> parts(G);
  for (int d = 0; d < G; ++d) {
    MultiPart& p = parts[d];
    p.device = devices[d];
    p.z0 = sz * d / G; p.zc = sz * (d + 1) / G - p.z0;
    p.y0 = sy * d / G; p.yc = sy * (d + 1) / G - p.y0;
  }
  MultiBarrier barrier;
  barrier.parties = G;
  const size_t row_l = (size_t)sx * label_bytes, row_f = (size_t)sx * sizeof(float);

  auto worker = [&](int d) -> int {
    MultiPart& me = parts[d];
    DeviceGuard restore_device;
    DeviceCache* dc = nullptr;
    int wrc = probe(me.device, &dc);
    std::unique_lock<std::mutex> host_call;
    auto note = [&](int code) { snprintf(me.error, sizeof(me.error), "device %d: %.200s", me.device, g_error); return code; };
    #define MULTI_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess && !wrc) { \
        wrc = fail(e_ == cudaErrorMemoryAllocation ? EDTB200_ENOMEM : EDTB200_ECUDA, "%s: %s", #expr, \
                   cudaGetErrorString(e_)); note(wrc); } } while (0)
    if (!wrc) {
      host_call = std::unique_lock<std::mutex>(dc->host_call);
      for (int o = 0; o < G; ++o)                                 // direct NVLink copies where possible
        if (o != d) { cudaDeviceEnablePeerAccess(parts[o].device, 0); cudaGetLastError(); }
      MULTI_TRY(ensure_stream(dc->stream));
      me.stream = dc->stream;
      MULTI_TRY(cudaEventCreateWithFlags(&me.after_y, cudaEventDisableTiming));
      MULTI_TRY(cudaEventCreateWithFlags(&me.after_z, cudaEventDisableTiming));
      const size_t nz_vox = (size_t)sx * sy * me.zc, ny_vox = (size_t)sx * me.yc * sz;
      MULTI_TRY(scratch_alloc(*dc, &me.lz, nz_vox * label_bytes, me.stream));
      MULTI_TRY(scratch_alloc(*dc, reinterpret_cast<void**>(&me.fz), nz_vox * sizeof(float), me.stream));
      MULTI_TRY(scratch_alloc(*dc, &me.ly, ny_vox * label_bytes, me.stream));
      MULTI_TRY(scratch_alloc(*dc, reinterpret_cast<void**>(&me.fy), ny_vox * sizeof(float), me.stream));
    } else {
      note(wrc);
    }
    // ---- phase A: my Z slab up, X and Y passes ----
    if (!wrc) {
      const char* src = static_cast<const char*>(labels) + (size_t)me.z0 * sy * row_l;
      wrc = upload(me.lz, src, (size_t)sx * sy * me.zc * label_bytes, me.device, me.stream);
      if (!wrc) wrc = first_pass(label_bytes, me.lz, me.fz, sy * me.zc, sx, wx, border, zero_label_flags(flags), *dc,
                                 me.stream);
      if (!wrc) wrc = later_pass(1, label_bytes, me.lz, me.fz, sx, sy, sz, me.zc, w, border, border, 0,
                                 /*pdl=*/true, *dc, me.stream);
      if (wrc) note(wrc);
      MULTI_TRY(cudaEventRecord(me.after_y, me.stream));
    }
    int agreed = barrier.arrive(wrc);
    // ---- phase B: gather my Y slab (whole z lines) from every Z slab, Z pass ----
    if (!agreed) {
      for (int o = 0; o < G && !wrc; ++o) {
        const MultiPart& src = parts[o];
        MULTI_TRY(cudaStreamWaitEvent(me.stream, src.after_y, 0));
        MULTI_TRY(copy_box(me.fy, row_f, me.yc, me.device, 0, 0, src.z0, src.fz, row_f, sy, src.device, 0, me.y0, 0,
                           row_f, me.yc, src.zc, me.stream));
        MULTI_TRY(copy_box(me.ly, row_l, me.yc, me.device, 0, 0, src.z0, src.lz, row_l, sy, src.device, 0, me.y0, 0,
                           row_l, me.yc, src.zc, me.stream));
      }
      if (!wrc) {
        wrc = later_pass(2, label_bytes, me.ly, me.fy, sx, sy, sz, me.yc, w, border, border, epilogue_flags(flags),
                         /*pdl=*/false, *dc, me.stream);
        if (wrc) note(wrc);
      }
      MULTI_TRY(cudaEventRecord(me.after_z, me.stream));
    }
    agreed = barrier.arrive(wrc);
    // ---- phase C: my Z slab of the result back from every Y slab, then down to the host ----
    if (!agreed) {
      for (int o = 0; o < G && !wrc; ++o) {
        const MultiPart& src = parts[o];
        MULTI_TRY(cudaStreamWaitEvent(me.stream, src.after_z, 0));
        MULTI_TRY(copy_box(me.fz, row_f, sy, me.device, 0, src.y0, 0, src.fy, row_f, src.yc, src.device, 0, 0, me.z0,
                           row_f, src.yc, me.zc, me.stream));
      }
      if (!wrc) {
        char* dst = reinterpret_cast<char*>(out) + (size_t)me.z0 * sy * row_f;
        wrc = download(dst, me.fz, (size_t)sx * sy * me.zc * sizeof(float), me.device, me.stream);
        if (wrc) note(wrc);
      }
    }
    if (me.stream) cudaStreamSynchronize(me.stream);
    agreed = barrier.arrive(wrc);                                 // nobody frees what a peer may still read
    void* all[] = {me.lz, me.fz, me.ly, me.fy};
    for (void* q : all) if (q) cudaFreeAsync(q, me.stream);
    if (me.after_y) cudaEventDestroy(me.after_y);
    if (me.after_z) cudaEventDestroy(me.after_z);
    cudaGetLastError();
    #undef MULTI_TRY
    return wrc ? wrc : agreed;
  };

  std::vector<int> rcs(G, 0);
  std::vector<std::thread> threads;
  for (int d = 1; d < G; ++d) threads.emplace_back([&, d] { rcs[d] = worker(d); });
  rcs[0] = worker(0);
  for (auto& t : threads) t.join();
  for (int d = 0; d < G; ++d)
    if (rcs[d] && parts[d].error[0]) return fail(rcs[d], "%s", parts[d].error);
  for (int d = 0; d < G; ++d)
    if (rcs[d]) return fail(rcs[d], "multi-device transform failed on device %d", parts[d].device);
  return 0;
}

int64_t edtb200_slab_stage_bytes(int64_t sx, int64_t sy, int label_bytes, int halo) {
  if (sx <= 0 || sy <= 0 || halo < 1 || halo > 254 ||
      !(label_bytes == 1 || label_bytes == 2 || label_bytes == 4 || label_bytes == 8))
    return -1;
  return (int64_t)edtb200::slab_stage_layout(sx * sy, label_bytes, halo).total_bytes;
}

int edtb200_slab_step(const void* labels_dev, int label_bytes, int64_t sx, int64_t sy, int64_t sz,
                      float wx, float wy, float wz, int black_border, int has_lo, int has_hi, int flags,
                      float* f_dev, int halo, void* sym_self, void* sym_lo, void* sym_hi,
                      unsigned long long step, int* status_dev, int device, void* stream_v) {
  using namespace edtb200;
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (halo < 1 || halo > 254) return fail(EDTB200_EINVAL, "halo must be in 1..254");
  if (sz <= halo && (has_lo || has_hi)) return fail(EDTB200_EINVAL, "the slab must be deeper than the halo");
  if (!labels_dev || !f_dev || !sym_self || !status_dev) return fail(EDTB200_EINVAL, "null pointer");
  if ((has_lo && !sym_lo) || (has_hi && !sym_hi)) return fail(EDTB200_EINVAL, "missing neighbour buffer");
  if (step == 0) return fail(EDTB200_EINVAL, "steps are counted from 1");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int border = black_border != 0;
  const int zero_label = zero_label_flags(flags);
  const int epilogue = epilogue_flags(flags);
  const float w[3] = {wx, wy, wz};

  // EDT_B200_VERBOSE=1: device time of every phase of the step on stderr (synchronises the stream)
  static const bool verbose = getenv("EDT_B200_VERBOSE") != nullptr && atoi(getenv("EDT_B200_VERBOSE")) != 0;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  auto stamp = [&](int i) {
    if (!verbose) return;
    if (cudaEventCreate(&ev[i]) == cudaSuccess) cudaEventRecord(ev[i], stream);
    cudaGetLastError();
  };
  stamp(0);
  mark_pass(0, stream);              // per-pass events for bench.py (edtb200_profile_passes), as in run_passes
  // X and Y passes: slab-local
  nvtx_push("edt.x");
  rc = first_pass(label_bytes, labels_dev, f_dev, sy * sz, sx, wx, border, zero_label, *dc, stream);
  nvtx_pop();
  if (rc) return rc;
  stamp(1);
  mark_pass(1, stream);
  nvtx_push("edt.y");
  rc = later_pass(1, label_bytes, labels_dev, f_dev, sx, sy, sz, sz, w, border, border, 0, /*pdl=*/!verbose, *dc,
                  stream);
  nvtx_pop();
  if (rc) return rc;
  stamp(2);

  const int64_t plane = sx * sy;
  const SlabStageLayout L = slab_stage_layout(plane, label_bytes, halo);
  unsigned char* self = static_cast<unsigned char*>(sym_self);
  unsigned char* lo = static_cast<unsigned char*>(sym_lo);
  unsigned char* hi = static_cast<unsigned char*>(sym_hi);
  const int parity = (int)(step & 1ull);
  const dim3 grid((unsigned)((plane + 255) / 256), 2);
  if (has_lo || has_hi) {
    nvtx_push("edt.halo.stage");
    unsigned char* set = self + (size_t)parity * L.set_bytes;
    // I am the HIGH neighbour of the rank below me and the LOW neighbour of the rank above me
    unsigned long long* flag_in_lo_peer = has_lo ? reinterpret_cast<unsigned long long*>(lo + L.flag_from_hi) : nullptr;
    unsigned long long* flag_in_hi_peer = has_hi ? reinterpret_cast<unsigned long long*>(hi + L.flag_from_lo) : nullptr;
    unsigned int* counter = reinterpret_cast<unsigned int*>(self + L.counter);
    with_label_width(label_bytes, [&](auto lw) {
      using LW = decltype(lw);
      slab_stage_kernel<LW::Bytes><<<grid, 256, 0, stream>>>(static_cast<const typename LW::T*>(labels_dev), f_dev,
                                                             plane, (int)sz, halo, has_lo, has_hi, set, L, step,
                                                             flag_in_lo_peer, flag_in_hi_peer, counter);
    });
    CUDA_TRY(cudaGetLastError());
    nvtx_pop();
  }

  stamp(3);
  mark_pass(2, stream);              // "second pass" = Y plus the face staging kernel
  // Z pass on the slab, interior faces open
  nvtx_push("edt.z");
  rc = later_pass(2, label_bytes, labels_dev, f_dev, sx, sy, sz, sy, w, border && !has_lo, border && !has_hi,
                  epilogue, /*pdl=*/!verbose && (has_lo || has_hi), *dc, stream);
  nvtx_pop();
  if (rc) return rc;

  stamp(4);
  mark_pass(3, stream);
  if (has_lo || has_hi) {
    nvtx_push("edt.halo.fixup");
    const int kflags = epilogue | zero_label;
    const float w2 = wz * wz;
    const unsigned char* set_lo = has_lo ? lo + (size_t)parity * L.set_bytes : nullptr;
    const unsigned char* set_hi = has_hi ? hi + (size_t)parity * L.set_bytes : nullptr;
    const unsigned long long* flag_from_lo = reinterpret_cast<const unsigned long long*>(self + L.flag_from_lo);
    const unsigned long long* flag_from_hi = reinterpret_cast<const unsigned long long*>(self + L.flag_from_hi);
    cudaLaunchAttribute fattr;
    fattr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    fattr.val.programmaticStreamSerializationAllowed = 1;
    // PDL behind our own Z pass, which triggers its dependents early
    const cudaLaunchConfig_t fcfg = {grid, dim3(256), 0, stream, &fattr, verbose ? 0u : 1u};
    CUDA_TRY(with_label_width(label_bytes, [&](auto lw) {
      using LW = decltype(lw);
      return cudaLaunchKernelEx(&fcfg, slab_fixup_kernel<LW::Bytes>, static_cast<const typename LW::T*>(labels_dev),
                                f_dev, plane, (int)sz, halo, w2, has_lo, has_hi, set_lo, set_hi, L, step, flag_from_lo,
                                flag_from_hi, kflags, status_dev);
    }));
    CUDA_TRY(cudaGetLastError());
    nvtx_pop();
  }
  stamp(5);
  if (verbose) {
    float ms[5] = {0, 0, 0, 0, 0};
    if (ev[5] && cudaEventSynchronize(ev[5]) == cudaSuccess)
      for (int i = 0; i < 5; ++i) if (ev[i] && ev[i + 1]) cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    fprintf(stderr, "[edt_b200] slab step %llu dev %d: x %.3f  y %.3f  stage %.3f  z %.3f  fixup %.3f ms\n", step, device,
            ms[0], ms[1], ms[2], ms[3], ms[4]);
    for (auto& e : ev) if (e) cudaEventDestroy(e);
    cudaGetLastError();
  }
  return 0;
}

int edtb200_label_stats(const void* labels_dev, int label_bytes, const float* dt_dev, int64_t sx, int64_t sy,
                        int64_t sz, int capacity, unsigned long long* keys_dev, unsigned long long* count_dev,
                        float* max_dev, long long* argmax_dev, int* box_dev, int* overflow_dev, int device,
                        void* stream_v) {
  using namespace edtb200;
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (capacity < 2 || (capacity & (capacity - 1))) return fail(EDTB200_EINVAL, "capacity must be a power of two");
  if (!labels_dev || !dt_dev || !keys_dev || !count_dev || !max_dev || !argmax_dev || !box_dev || !overflow_dev)
    return fail(EDTB200_EINVAL, "null pointer");
  if (sx > 0x7fffffff || sy > 0x7fffffff || sz > 0x7fffffff) return fail(EDTB200_ELIMIT, "axis too long");
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  LabelTable t;
  t.keys = keys_dev; t.count = count_dev; t.maxbits = reinterpret_cast<unsigned int*>(max_dev);
  t.argmax = argmax_dev; t.box = box_dev; t.capacity = capacity; t.overflow = overflow_dev;
  label_table_init_kernel<<<(capacity + 255) / 256, 256, 0, stream>>>(t);
  CUDA_TRY(cudaMemsetAsync(overflow_dev, 0, sizeof(int), stream));
  const int64_t total = sx * sy * sz;
  if (total > 0) {
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)dc->sm_count * 16);
    with_label_width(label_bytes, [&](auto lw) {
      using LW = decltype(lw);
      const auto* lab = static_cast<const typename LW::T*>(labels_dev);
      label_stats_kernel<LW::Bytes><<<blocks, 256, 0, stream>>>(lab, dt_dev, total, (int)sx, (int)sy, t);
      label_argmax_kernel<LW::Bytes><<<blocks, 256, 0, stream>>>(lab, dt_dev, total, t);
    });
  }
  label_table_finish_kernel<<<(capacity + 255) / 256, 256, 0, stream>>>(t);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int edtb200_label_extract(const void* labels_dev, int label_bytes, const float* dt_dev, int64_t sx, int64_t sy,
                          int64_t sz, unsigned long long key, const int* box, int erase, float* out_dev,
                          int device, void* stream_v) {
  using namespace edtb200;
  int rc = check_dims(label_bytes, 3, sx, sy, sz);
  if (rc) return rc;
  if (!labels_dev || !dt_dev || !out_dev) return fail(EDTB200_EINVAL, "null pointer");
  if (sx > 0x7fffffff || sy > 0x7fffffff || sz > 0x7fffffff) return fail(EDTB200_ELIMIT, "axis too long");
  int b[6] = {0, 0, 0, (int)sx - 1, (int)sy - 1, (int)sz - 1};
  if (box) for (int i = 0; i < 6; ++i) b[i] = box[i];
  if (b[0] < 0 || b[1] < 0 || b[2] < 0 || b[3] >= sx || b[4] >= sy || b[5] >= sz)
    return fail(EDTB200_EINVAL, "box outside the volume");
  if (b[3] < b[0] || b[4] < b[1] || b[5] < b[2]) return 0;             // empty box
  DeviceGuard restore_device;
  DeviceCache* dc = nullptr;
  rc = probe(device, &dc);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int bx = b[3] - b[0] + 1, by = b[4] - b[1] + 1, bz = b[5] - b[2] + 1;
  const int64_t rows = (int64_t)by * bz;
  const unsigned blocks = (unsigned)std::min<int64_t>((rows + 7) / 8, (int64_t)dc->sm_count * 16);
  with_label_width(label_bytes, [&](auto lw) {
    using LW = decltype(lw);
    label_extract_kernel<LW::Bytes><<<blocks, 256, 0, stream>>>(static_cast<const typename LW::T*>(labels_dev), dt_dev,
                                                                out_dev, (int)sx, (int)sy, b[0], b[1], b[2], bx, by,
                                                                bz, key, erase);
  });
  CUDA_TRY(cudaGetLastError());
  return 0;
}

void* edtb200_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void edtb200_host_free(void* p) {
  if (p) { cudaFreeHost(p); cudaGetLastError(); }
}

int edtb200_profile_passes(int enable) {
  g_profile = enable != 0;
  if (enable) g_pass_seq = 0;
  return 0;
}

int edtb200_pass_ms(int steps_back, float* ms3) {
  if (!ms3) return fail(EDTB200_EINVAL, "null pointer");
  ms3[0] = ms3[1] = ms3[2] = 0.0f;
  if (steps_back < 0 || steps_back >= kProfileRing || steps_back >= g_pass_seq)
    return fail(EDTB200_EINVAL, "no profiled transform %d steps back", steps_back);
  const int slot = (int)((g_pass_seq - 1 - steps_back) % kProfileRing);
  for (int i = 0; i < g_pass_marks[slot] && i < 3; ++i) {
    if (!g_pass_events[slot][i] || !g_pass_events[slot][i + 1]) break;
    CUDA_TRY(cudaEventSynchronize(g_pass_events[slot][i + 1]));
    CUDA_TRY(cudaEventElapsedTime(&ms3[i], g_pass_events[slot][i], g_pass_events[slot][i + 1]));
  }
  return 0;
}

int edtb200_release(void) {
  DeviceGuard restore_device;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
  for (int d = 0; d < count && d < kMaxDevices; ++d) {
    DeviceCache& dc = g_cache[d];
    std::lock_guard<std::mutex> host_call(dc.host_call);
    std::lock_guard<std::mutex> guard(dc.lock);
    if (!dc.probed) continue;
    cudaSetDevice(d);
    cudaDeviceSynchronize();
    for (auto& t : dc.tables) {
      if (t.data) cudaFree(t.data);
      if (t.ready) cudaEventDestroy(t.ready);
      for (auto& e : t.used) if (e) cudaEventDestroy(e);
      t = DeviceCache::Table();
    }
    if (dc.stream) { cudaStreamSynchronize(dc.stream); cudaStreamDestroy(dc.stream); }
    if (dc.labels) cudaFree(dc.labels);
    if (dc.dist) cudaFree(dc.dist);
    if (dc.labels2) cudaFree(dc.labels2);
    if (dc.dist2) cudaFree(dc.dist2);
    if (dc.stream_up) cudaStreamDestroy(dc.stream_up);
    if (dc.stream_down) cudaStreamDestroy(dc.stream_down);
    for (int i = 0; i < 2; ++i) {
      if (dc.ev_up[i]) cudaEventDestroy(dc.ev_up[i]);
      if (dc.ev_comp[i]) cudaEventDestroy(dc.ev_comp[i]);
      if (dc.ev_down[i]) cudaEventDestroy(dc.ev_down[i]);
    }
    dc.labels = dc.labels2 = nullptr; dc.dist = dc.dist2 = nullptr;
    dc.labels_bytes = dc.labels2_bytes = dc.dist_bytes = dc.dist2_bytes = 0;
    dc.stream = dc.stream_up = dc.stream_down = nullptr;
    for (int i = 0; i < 2; ++i) dc.ev_up[i] = dc.ev_comp[i] = dc.ev_down[i] = nullptr;
    // everything the stream-ordered scratch pool still holds goes back to the driver
    if (dc.pool) cudaMemPoolTrimTo(dc.pool, 0);
    for (int dir = 0; dir < 2; ++dir) {
      StageBuffers& sb = g_stage[dir][d];
      for (int i = 0; i < kStages; ++i) {
        if (sb.buf[i]) { cudaFreeHost(sb.buf[i]); sb.buf[i] = nullptr; }
        if (sb.ev[i]) { cudaEventDestroy(sb.ev[i]); sb.ev[i] = nullptr; }
      }
    }
    cudaGetLastError();
  }
  return 0;
}

}  // extern "C"
