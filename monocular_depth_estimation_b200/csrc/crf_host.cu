// Host-side plumbing of libcrf_sm100.so: thread-local error string, TMA descriptor creation.
#include "crf_host.h"

#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace crf {

namespace {
thread_local char g_err[512] = "";
}

int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
const char* get_error() { return g_err; }

namespace {
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_encode_once;

void load_encode() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
      q == cudaDriverEntryPointSuccess)
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
}
}  // namespace

int make_tmap_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  std::call_once(g_encode_once, load_encode);
  CRF_CHECK(g_encode != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  CRF_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA: base pointer %p is not 16-byte aligned", ptr);
  CRF_CHECK(cols % 4 == 0, "TMA: row pitch must be a multiple of 16 bytes (cols=%llu)", (unsigned long long)cols);
  CRF_CHECK(box_rows >= 1 && box_rows <= 256, "TMA: box rows %u out of range", box_rows);
  const cuuint64_t gdim[2] = {cols, rows};
  const cuuint64_t gstride[1] = {cols * 4};
  const cuuint32_t box[2] = {32, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), gdim, gstride, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CRF_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(f32) failed: %d (rows=%llu cols=%llu box_rows=%u)", (int)r,
            (unsigned long long)rows, (unsigned long long)cols, box_rows);
  return 0;
}

int make_tmap_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  std::call_once(g_encode_once, load_encode);
  CRF_CHECK(g_encode != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  CRF_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA: base pointer %p is not 16-byte aligned", ptr);
  CRF_CHECK(cols % 8 == 0, "TMA: row pitch must be a multiple of 16 bytes (cols=%llu)", (unsigned long long)cols);
  CRF_CHECK(box_rows >= 1 && box_rows <= 256, "TMA: box rows %u out of range", box_rows);
  const cuuint64_t gdim[2] = {cols, rows};
  const cuuint64_t gstride[1] = {cols * 2};
  const cuuint32_t box[2] = {64, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CRF_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed: %d (rows=%llu cols=%llu box_rows=%u)", (int)r,
            (unsigned long long)rows, (unsigned long long)cols, box_rows);
  return 0;
}

namespace {
std::atomic<long long> g_launches{0};
}
void note_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---- per-kernel timing --------------------------------------------------------------------------
namespace {
struct TimingEntry {
  double flops = 0, bytes = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> evs;
};
std::mutex g_tm_mu;
std::atomic<bool> g_timing{false};
std::map<std::string, TimingEntry> g_tm;
}  // namespace

KernelTimer::KernelTimer(cudaStream_t st, double flops, double bytes, const char* fmt, ...)
    : st_(st), flops_(flops), bytes_(bytes) {
  if (!g_timing.load(std::memory_order_relaxed)) return;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(label_, sizeof(label_), fmt, ap);
  va_end(ap);
  if (cudaEventCreate(&e0_) != cudaSuccess || cudaEventCreate(&e1_) != cudaSuccess) return;
  on_ = true;
  cudaEventRecord(e0_, st_);
}
KernelTimer::~KernelTimer() {
  if (!on_) return;
  cudaEventRecord(e1_, st_);
  std::lock_guard<std::mutex> lk(g_tm_mu);
  TimingEntry& e = g_tm[label_];
  e.flops = flops_;
  e.bytes = bytes_;
  e.evs.emplace_back(e0_, e1_);
}
void timing_enable(bool on) {
  std::lock_guard<std::mutex> lk(g_tm_mu);
  if (on) {
    for (auto& kv : g_tm)
      for (auto& p : kv.second.evs) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    g_tm.clear();
  }
  g_timing.store(on);
}
// JSON array: [{"kernel": label, "launches": n, "total_ms": t, "flops": per-launch, "bytes": per-launch}, ...]
size_t timing_report(char* buf, size_t cap) {
  std::lock_guard<std::mutex> lk(g_tm_mu);
  std::string out = "[";
  bool first = true;
  for (auto& kv : g_tm) {
    double total = 0;
    for (auto& p : kv.second.evs) {
      cudaEventSynchronize(p.second);
      float ms = 0;
      if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) total += ms;
    }
    char line[320];
    snprintf(line, sizeof(line), "%s{\"kernel\": \"%s\", \"launches\": %zu, \"total_ms\": %.6f, \"flops\": %.6e, \"bytes\": %.6e}",
             first ? "" : ", ", kv.first.c_str(), kv.second.evs.size(), total, kv.second.flops, kv.second.bytes);
    out += line;
    first = false;
  }
  out += "]";
  if (buf != nullptr && cap > 0) {
    const size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return out.size() + 1;
}

int num_sms(int device) {
  static int cached[64] = {0};
  if (device < 0 || device >= 64) return 148;
  if (cached[device] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
    cached[device] = n;
  }
  return cached[device];
}

}  // namespace crf
