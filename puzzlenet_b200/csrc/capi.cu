// Library-wide pieces of the C ABI (include/puzzlenet_b200.h): version, error text, device probe.
#include <atomic>
#include <mutex>
#include <vector>

#include "pz_common.cuh"

namespace pz {

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

// ---- launch counter -------------------------------------------------------------------
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// ---- stage profiler: event sets, one per profiled call ----------------------------------
constexpr int PROF_MAX_SETS = 512, PROF_MAX_MARKS = 48;
struct ProfSet {
  cudaEvent_t ev[PROF_MAX_MARKS + 1];
  const char* name[PROF_MAX_MARKS + 1];
  int lane[PROF_MAX_MARKS + 1];
  int n = 0;
  bool created = false;
};
static bool g_prof_on = false;
static bool g_prof_serial = false;
static std::vector<ProfSet>* g_sets = nullptr;
static int g_cur = -1;
static std::mutex g_prof_mu;

void prof_begin(cudaStream_t st) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_sets) g_sets = new std::vector<ProfSet>(PROF_MAX_SETS);
  if (g_cur + 1 >= PROF_MAX_SETS) { g_cur = PROF_MAX_SETS; return; }
  ProfSet& s = (*g_sets)[++g_cur];
  if (!s.created) {
    for (auto& e : s.ev) cudaEventCreate(&e);
    s.created = true;
  }
  s.n = 0;
  s.name[0] = "_begin";
  s.lane[0] = 0;
  cudaEventRecord(s.ev[0], st);
}
void prof_mark(const char* stage, cudaStream_t st, int lane) {
  if (!g_prof_on || !g_sets || g_cur < 0 || g_cur >= PROF_MAX_SETS) return;
  ProfSet& s = (*g_sets)[g_cur];
  if (s.n >= PROF_MAX_MARKS) return;
  ++s.n;
  s.name[s.n] = stage;
  s.lane[s.n] = lane;
  cudaEventRecord(s.ev[s.n], st);
}

bool prof_serial() { return g_prof_serial; }
bool pdl_for_stream(cudaStream_t st) {
  if (g_prof_on) return false;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return cs == cudaStreamCaptureStatusNone;
}

// One side stream + event set per (device, caller stream): two host threads that enqueue on different streams of the
// same device never share fork/join events (a shared set lets one call's geometry wait on the other call's fork), and
// concurrent callers do not serialise their geometry on one stream.  Calls on the SAME caller stream are ordered by that
// stream, as in any CUDA API.  The table is bounded: past 256 distinct caller streams the oldest entry is recycled
// (its events are only ever waited on by work enqueued before the recycling call returns).
int side_stream(SideStream** out, cudaStream_t caller) {
  struct Entry {
    int dev = -1;
    cudaStream_t caller = nullptr;
    SideStream s;
  };
  static std::mutex mu;
  static std::vector<Entry>* table = nullptr;
  static size_t next_victim = 0;
  int dev = 0;
  PZ_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (!table) {
    table = new std::vector<Entry>();
    table->reserve(256);          // entries never move: callers keep SideStream* across the lock
  }
  for (Entry& e : *table)
    if (e.dev == dev && e.caller == caller) {
      *out = &e.s;
      return 0;
    }
  Entry* e = nullptr;
  if (table->size() < 256) {
    table->emplace_back();
    e = &table->back();
    PZ_CUDA(cudaStreamCreateWithFlags(&e->s.stream, cudaStreamNonBlocking));
    PZ_CUDA(cudaEventCreateWithFlags(&e->s.fork, cudaEventDisableTiming));
    PZ_CUDA(cudaEventCreateWithFlags(&e->s.join, cudaEventDisableTiming));
  } else {
    for (size_t tries = 0; tries < table->size() && !e; ++tries) {   // recycle an entry of the same device
      Entry& c = (*table)[next_victim++ % table->size()];
      if (c.dev == dev) e = &c;
    }
    PZ_REQUIRE(e != nullptr, PZ_ERR_UNSUPPORTED, "side_stream: stream table exhausted");
  }
  e->dev = dev;
  e->caller = caller;
  *out = &e->s;
  return 0;
}

}  // namespace pz

extern "C" long long pz_launch_count(void) { return pz::g_launches.load(); }

extern "C" int pz_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(pz::g_prof_mu);
  pz::g_prof_on = on != 0;
  pz::g_prof_serial = on == 2;
  pz::g_cur = -1;
  return 0;
}

// Sums, over every profiled call since pz_profile_enable(1), the elapsed ms of each stage (stages are
// keyed by position; names[i] receives a static string).  Synchronises the device.  Returns the stage count.
extern "C" int pz_profile_collect(double* ms, const char** names, int* calls, int max_stages) {
  std::lock_guard<std::mutex> lk(pz::g_prof_mu);
  if (calls) *calls = 0;
  if (!pz::g_sets || pz::g_cur < 0) return 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return pz::fail(-1000, "pz_profile_collect: device sync failed");
  const int nsets = pz::g_cur < pz::PROF_MAX_SETS ? pz::g_cur + 1 : pz::PROF_MAX_SETS;
  int nstage = 0;
  for (int i = 0; i < max_stages; ++i) ms[i] = 0.0;
  for (int c = 0; c < nsets; ++c) {
    pz::ProfSet& s = (*pz::g_sets)[c];
    int last[2] = {0, -1};
    for (int i = 1; i <= s.n && i <= max_stages; ++i) {
      const int lane = s.lane[i] & 1;
      float t = 0.f;
      if (last[lane] >= 0 && s.name[i][0] != '_') cudaEventElapsedTime(&t, s.ev[last[lane]], s.ev[i]);
      last[lane] = i;
      ms[i - 1] += t;
      if (names) names[i - 1] = s.name[i];
    }
    if (s.n > nstage) nstage = s.n;
  }
  if (calls) *calls = nsets;
  pz::g_cur = -1;
  return nstage < max_stages ? nstage : max_stages;
}

extern "C" int pz_abi_version(void) { return PZ_ABI_VERSION; }

extern "C" const char* pz_last_error(void) { return pz::error_buffer(); }

extern "C" int pz_device_arch(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return pz::fail(-1000, "cudaGetDevice failed (no CUDA device?)");
  int major = 0, minor = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess)
    return pz::fail(-1000, "cudaDeviceGetAttribute failed");
  return major * 10 + minor;
}
