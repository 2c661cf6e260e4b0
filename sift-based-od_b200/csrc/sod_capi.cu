// Library-wide pieces of the C ABI: version, error string, device query.
#include <cstring>

#include "sod_common.cuh"

namespace sod {

namespace {
thread_local char g_err[512] = {0};
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- stage timers: a ring of event pairs per stage, filled while enabled, drained by sod_timing_read
namespace {
constexpr int kTimerRing = 128;
struct StageTimers {
  bool on = false;
  cudaEvent_t ev[SOD_STAGE_COUNT][kTimerRing][2] = {};
  int head[SOD_STAGE_COUNT] = {};   // pairs recorded since the last read
  bool open[SOD_STAGE_COUNT] = {};
};
thread_local StageTimers g_timers;
}  // namespace

void stage_begin(int stage, cudaStream_t st) {
  StageTimers& t = g_timers;
  if (!t.on || stage < 0 || stage >= SOD_STAGE_COUNT || t.head[stage] >= kTimerRing) return;
  cudaEvent_t& e = t.ev[stage][t.head[stage]][0];
  if (!e && cudaEventCreate(&e) != cudaSuccess) return;
  t.open[stage] = cudaEventRecord(e, st) == cudaSuccess;
}

void stage_end(int stage, cudaStream_t st) {
  StageTimers& t = g_timers;
  if (!t.on || stage < 0 || stage >= SOD_STAGE_COUNT || !t.open[stage]) return;
  t.open[stage] = false;
  cudaEvent_t& e = t.ev[stage][t.head[stage]][1];
  if (!e && cudaEventCreate(&e) != cudaSuccess) return;
  if (cudaEventRecord(e, st) == cudaSuccess) ++t.head[stage];
}

int device_sm_count() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    set_error("cannot query the current CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    return -1;
  }
  return sms;
}

}  // namespace sod

extern "C" {

int sod_version(void) { return 2000; }

const char* sod_last_error(void) { return sod::g_err; }

int sod_device_sm_count(void) { return sod::device_sm_count(); }

int sod_timing_enable(int32_t on) {
  sod::g_timers.on = on != 0;
  for (int s = 0; s < SOD_STAGE_COUNT; ++s) {
    sod::g_timers.head[s] = 0;
    sod::g_timers.open[s] = false;
  }
  return SOD_OK;
}

int32_t sod_timing_read(int32_t stage, float* ms_host, int32_t cap) {
  sod::StageTimers& t = sod::g_timers;
  if (stage < 0 || stage >= SOD_STAGE_COUNT || (cap > 0 && !ms_host)) {
    sod::set_error("sod_timing_read: bad stage or null buffer");
    return SOD_ERR_INVALID_ARGUMENT;
  }
  const int n = t.head[stage];
  int out = 0;
  for (int i = 0; i < n; ++i) {
    float ms = 0.f;
    if (cudaEventSynchronize(t.ev[stage][i][1]) != cudaSuccess ||
        cudaEventElapsedTime(&ms, t.ev[stage][i][0], t.ev[stage][i][1]) != cudaSuccess) {
      sod::set_error("sod_timing_read: %s", cudaGetErrorString(cudaGetLastError()));
      t.head[stage] = 0;
      return SOD_ERR_CUDA;
    }
    if (out < cap) ms_host[out++] = ms;
  }
  t.head[stage] = 0;
  return out;
}

}  // extern "C"
