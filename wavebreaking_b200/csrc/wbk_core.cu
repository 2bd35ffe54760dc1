// Error plumbing and library-level entry points of libwbk.
#include "wbk_common.cuh"
#include <cstdarg>

static thread_local char g_err[512] = "";

void wbk_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* wbk_last_error(void) { return g_err; }

extern "C" int wbk_version(void) { return 100; }

extern "C" int wbk_device_count(void) {
#ifdef WBK_EMU
  return 1;
#else
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    wbk_set_error("no CUDA device available (%s); libwbk has no CPU path", e != cudaSuccess ? cudaGetErrorString(e) : "count == 0");
    return WBK_ERR_NODEVICE;
  }
  return n;
#endif
}

// ------------------------------------------------------------------------------------------ profiler
#include <atomic>
#include <mutex>
#include <vector>

static const char* kKernelNames[WBK_PROF_NKERNELS] = {
    "smooth_fused", "convolve2d", "nan_border", "mflux", "flip", "synth_pv", "ms_segments", "contour_link",
    "contours_pack", "select", "overturning", "streamer_prep", "tile_scan", "pair_scan", "streamer_dedupe",
    "event_list", "events_raster", "rings_raster", "owner", "events_gather", "track_overlap", "misc", "split_events",
    "split_raster", "streamer_touch", "streamer_finish", "smooth_ms_fused", "track_pairs", "track_exact", "track_distance",
    "flag_counts", "track_append"};

static std::atomic<long long> g_launches{0};
static std::atomic<int> g_prof_on{0};

#ifndef WBK_EMU
namespace {
struct ProfRec {
  int kid;
  cudaEvent_t a, b;
};
std::mutex g_prof_mu;
std::vector<ProfRec> g_recs;
std::vector<cudaEvent_t> g_pool;
cudaEvent_t g_pending = nullptr;
double g_ms[WBK_PROF_NKERNELS];
int g_n[WBK_PROF_NKERNELS];

cudaEvent_t take_event() {
  if (!g_pool.empty()) {
    cudaEvent_t e = g_pool.back();
    g_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
void drain_locked() {
  for (auto& r : g_recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      g_ms[r.kid] += ms;
      g_n[r.kid] += 1;
    }
    g_pool.push_back(r.a);
    g_pool.push_back(r.b);
  }
  g_recs.clear();
}
}  // namespace
#endif

void wbk_prof_begin(int kid, void* stream) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
#ifndef WBK_EMU
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_pending = take_event();
  cudaEventRecord(g_pending, (cudaStream_t)stream);
#else
  (void)kid; (void)stream;
#endif
}

void wbk_prof_end(int kid, void* stream) {
#ifndef WBK_EMU
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_pending) return;
  ProfRec r;
  r.kid = kid;
  r.a = g_pending;
  r.b = take_event();
  g_pending = nullptr;
  cudaEventRecord(r.b, (cudaStream_t)stream);
  g_recs.push_back(r);
  if (g_recs.size() > 8192) drain_locked();
#else
  (void)kid; (void)stream;
#endif
}

extern "C" int wbk_prof_enable(int on) {
  g_prof_on.store(on ? 1 : 0);
  return WBK_OK;
}

extern "C" int wbk_prof_reset(void) {
#ifndef WBK_EMU
  std::lock_guard<std::mutex> lk(g_prof_mu);
  drain_locked();
  for (int k = 0; k < WBK_PROF_NKERNELS; ++k) {
    g_ms[k] = 0.0;
    g_n[k] = 0;
  }
#endif
  return WBK_OK;
}

extern "C" int wbk_prof_read(int* h_launches, double* h_ms) {
  if (!h_launches || !h_ms) {
    wbk_set_error("wbk_prof_read: invalid argument");
    return WBK_ERR_INVALID;
  }
#ifndef WBK_EMU
  std::lock_guard<std::mutex> lk(g_prof_mu);
  drain_locked();
  for (int k = 0; k < WBK_PROF_NKERNELS; ++k) {
    h_launches[k] = g_n[k];
    h_ms[k] = g_ms[k];
  }
#else
  for (int k = 0; k < WBK_PROF_NKERNELS; ++k) {
    h_launches[k] = 0;
    h_ms[k] = 0.0;
  }
#endif
  return WBK_OK;
}

extern "C" const char* wbk_prof_name(int k) { return (k >= 0 && k < WBK_PROF_NKERNELS) ? kKernelNames[k] : ""; }

extern "C" long long wbk_launch_count(void) { return g_launches.load(); }
