// Error reporting, launch counting and the optional per-kernel CUDA-event profiler of the C ABI.
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace hipac {
static thread_local std::string g_last_error;
static thread_local long long g_launches = 0;
void set_error(const std::string& msg) { g_last_error = msg; }
void count_launch(int n) { g_launches += n; }

int ensure_dyn_smem_impl(const void* func, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, int> done;   // (kernel, device) -> bytes already opted in
  int dev = 0;
  HIPAC_CHECK_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  auto it = done.find({func, dev});
  if (it != done.end() && it->second >= bytes) return 0;
  HIPAC_CHECK_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done[{func, dev}] = bytes;
  return 0;
}

int device_sm_count(int* sms) {
  static std::mutex mu;
  static int cache[64] = {};
  int dev = 0;
  HIPAC_CHECK_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (dev < 64 && cache[dev]) {
    *sms = cache[dev];
    return 0;
  }
  int n = 0;
  HIPAC_CHECK_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  if (dev < 64) cache[dev] = n;
  *sms = n;
  return 0;
}

// ---- profiler: cudaEvent pairs recorded on the launching stream around each kernel -------------
struct ProfRecord {
  const char* name;
  double work;  // algorithmic bytes or flops of this launch (0 if not stated)
  cudaEvent_t start, stop;
};
static thread_local bool g_prof_on = false;
static thread_local std::vector<ProfRecord> g_prof;
static thread_local std::vector<cudaEvent_t> g_event_pool;

static cudaEvent_t get_event() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

ProfileScope::ProfileScope(const char* name, cudaStream_t stream, double work) : idx_(-1), stream_(stream) {
  if (!g_prof_on) return;
  ProfRecord r{name, work, get_event(), get_event()};
  cudaEventRecord(r.start, stream);
  g_prof.push_back(r);
  idx_ = (int)g_prof.size() - 1;
}
ProfileScope::~ProfileScope() {
  if (idx_ >= 0) cudaEventRecord(g_prof[idx_].stop, stream_);
}
}  // namespace hipac

using namespace hipac;

extern "C" const char* hipac_last_error(void) { return g_last_error.c_str(); }
extern "C" int hipac_abi_version(void) { return HIPAC_ABI_VERSION; }
extern "C" long long hipac_launch_count(int reset) {
  long long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

extern "C" int hipac_profile_enable(int on) {
  g_prof_on = on != 0;
  return 0;
}

// Synchronises the recorded events and writes one line per kernel name:
//   "<name> <launches> <total_ms> <total_work>\n"   (work = algorithmic bytes or flops, 0 if unknown)
// Clears the records.  Returns the number of bytes the full report needs (excluding the NUL).
extern "C" long long hipac_profile_report(char* buf, size_t cap) {
  struct Acc { long long n = 0; double ms = 0, work = 0; };
  std::map<std::string, Acc> acc;
  std::vector<std::string> order;
  for (auto& r : g_prof) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.stop) == cudaSuccess) cudaEventElapsedTime(&ms, r.start, r.stop);
    if (!acc.count(r.name)) order.push_back(r.name);
    Acc& a = acc[r.name];
    a.n++, a.ms += ms, a.work += r.work;
    g_event_pool.push_back(r.start);
    g_event_pool.push_back(r.stop);
  }
  g_prof.clear();
  std::string out;
  for (auto& k : order) {
    char line[256];
    snprintf(line, sizeof line, "%s %lld %.6f %.6e\n", k.c_str(), acc[k].n, acc[k].ms, acc[k].work);
    out += line;
  }
  if (buf && cap) {
    size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return (long long)out.size();
}
