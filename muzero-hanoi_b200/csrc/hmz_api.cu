// Process-level plumbing of libhmz.so: error strings, launch counter, device queries.
#include <mutex>
#include <vector>

#include "hmz_common.cuh"

namespace hmz {

std::atomic<int> g_prof_on{0};
namespace {
struct ProfRec {
  int cls;
  cudaEvent_t start, stop;
};
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof;
}  // namespace

void prof_push(int cls, cudaStream_t stream, bool start) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (start) {
    ProfRec r{cls, nullptr, nullptr};
    if (cudaEventCreate(&r.start) != cudaSuccess || cudaEventCreate(&r.stop) != cudaSuccess) return;
    cudaEventRecord(r.start, stream);
    g_prof.push_back(r);
  } else {
    // the matching record is the most recent one of this class (scopes of one class do not nest)
    for (size_t i = g_prof.size(); i-- > 0;)
      if (g_prof[i].cls == cls) {
        cudaEventRecord(g_prof[i].stop, stream);
        break;
      }
  }
}

std::atomic<long long> g_launches{0};

char* error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 512, fmt, ap);
  va_end(ap);
  return code;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = kSmFallback;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return kSmFallback;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) cached = n;
    cached_dev = dev;
  }
  return cached;
}

// ---- launch Gantt recorder (tooling) ----
namespace {
constexpr int kGanttSlots = 16384;
std::mutex g_gantt_mu;
unsigned long long* g_gantt_dev = nullptr;
int g_gantt_on = 0, g_gantt_used = 0;
int g_gantt_meta[kGanttSlots][2];
thread_local int tl_gantt_tag = 0;
}  // namespace
unsigned long long* gantt_next(int kind, int tag) {
  if (!g_gantt_on) return nullptr;
  std::lock_guard<std::mutex> lk(g_gantt_mu);
  if (!g_gantt_on || g_gantt_used >= kGanttSlots) return nullptr;
  g_gantt_meta[g_gantt_used][0] = kind;
  g_gantt_meta[g_gantt_used][1] = tag;
  return g_gantt_dev + 2 * (size_t)(g_gantt_used++);
}
void gantt_set_context(int group, int sim) { tl_gantt_tag = (sim << 8) | (group & 0xFF); }
int gantt_context_tag() { return tl_gantt_tag; }

}  // namespace hmz

extern "C" {

// enable = 1: start recording (slots reset).  enable = 0: stop, synchronise the device and copy out up to max_records
// records of four words {kind (0 = network, 1 = tree), tag = sim << 8 | group, start ns, end ns}; *n_out = records written.
int hmz_debug_gantt(int enable, unsigned long long* host_out, int max_records, int* n_out) {
  using namespace hmz;
  std::lock_guard<std::mutex> lk(g_gantt_mu);
  if (enable) {
    if (!g_gantt_dev && cudaMalloc(&g_gantt_dev, sizeof(unsigned long long) * 2 * kGanttSlots) != cudaSuccess)
      return fail(HMZ_ERR_CUDA, "hmz_debug_gantt: cudaMalloc failed");
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemset(g_gantt_dev, 0xFF, sizeof(unsigned long long) * 2 * kGanttSlots) != cudaSuccess)
      return fail(HMZ_ERR_CUDA, "hmz_debug_gantt: reset failed");
    g_gantt_used = 0;
    g_gantt_on = 1;
    return HMZ_OK;
  }
  g_gantt_on = 0;
  if (n_out) *n_out = 0;
  if (!g_gantt_dev || !host_out) return HMZ_OK;
  if (cudaDeviceSynchronize() != cudaSuccess) return fail(HMZ_ERR_CUDA, "hmz_debug_gantt: synchronise failed");
  const int n = g_gantt_used < max_records ? g_gantt_used : max_records;
  std::vector<unsigned long long> raw(2 * (size_t)(n > 0 ? n : 1));
  if (n > 0 && cudaMemcpy(raw.data(), g_gantt_dev, sizeof(unsigned long long) * 2 * n, cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "hmz_debug_gantt: copy failed");
  for (int i = 0; i < n; ++i) {
    host_out[4 * i] = (unsigned long long)g_gantt_meta[i][0];
    host_out[4 * i + 1] = (unsigned long long)g_gantt_meta[i][1];
    host_out[4 * i + 2] = raw[2 * i];
    host_out[4 * i + 3] = ~raw[2 * i + 1];
  }
  if (n_out) *n_out = n;
  return HMZ_OK;
}

const char* hmz_last_error(void) { return hmz::error_buffer(); }

int hmz_version(void) { return 204; }

int64_t hmz_launch_count(void) { return (int64_t)hmz::g_launches.load(); }

int hmz_prof_begin(void) {
  std::lock_guard<std::mutex> lk(hmz::g_prof_mu);
  for (auto& r : hmz::g_prof) {
    cudaEventDestroy(r.start);
    cudaEventDestroy(r.stop);
  }
  hmz::g_prof.clear();
  hmz::g_prof_on.store(1);
  return HMZ_OK;
}

int hmz_prof_end(double* ms_by_class, int64_t* launches_by_class) {
  hmz::g_prof_on.store(0);
  std::lock_guard<std::mutex> lk(hmz::g_prof_mu);
  for (int c = 0; c < HMZ_PROF_CLASSES; ++c) {
    if (ms_by_class) ms_by_class[c] = 0.0;
    if (launches_by_class) launches_by_class[c] = 0;
  }
  int rc = HMZ_OK;
  for (auto& r : hmz::g_prof) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(r.stop);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.start, r.stop);
    if (e != cudaSuccess) rc = hmz::fail(HMZ_ERR_CUDA, "hmz_prof_end: %s", cudaGetErrorString(e));
    if (r.cls >= 0 && r.cls < HMZ_PROF_CLASSES) {
      if (ms_by_class) ms_by_class[r.cls] += ms;
      if (launches_by_class) launches_by_class[r.cls] += 1;
    }
    cudaEventDestroy(r.start);
    cudaEventDestroy(r.stop);
  }
  hmz::g_prof.clear();
  return rc;
}

int hmz_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return hmz::fail(HMZ_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp p;
  e = cudaGetDeviceProperties(&p, dev);
  if (e != cudaSuccess) return hmz::fail(HMZ_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  return HMZ_OK;
}

}  // extern "C"
