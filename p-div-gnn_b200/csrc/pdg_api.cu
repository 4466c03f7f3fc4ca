// Library-wide state: last-error string, version, SM count.
#include <atomic>
#include <mutex>
#include <stdarg.h>
#include <stdlib.h>
#include <vector>

#include "pdg_common.cuh"

namespace pdg {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int set_smem(const void* fn, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(%zu B smem): %s", bytes, cudaGetErrorString(e));
    return -2;
  }
  return 0;
}
int num_sms() {
  static int sms[64] = {0};
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  std::lock_guard<std::mutex> lk(mu);
  if (sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    sms[dev] = v;
  }
  return sms[dev];
}

bool pdl_enabled() {
  static const bool on = getenv("PDG_NO_PDL") == nullptr;
  return on;
}

static std::atomic<long long> g_launches{0};
void count_launches(int n) { g_launches += n; }

// ---- optional per-kernel-class CUDA-event timers (bench.py roofline) ----------------------
struct TimingRec { cudaEvent_t a, b; int cls; };
static std::mutex g_tmu;
static bool g_timing = false;
static std::vector<TimingRec> g_recs;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_pool;
void timing_begin(int cls, cudaStream_t st) {
  if (!g_timing) return;
  std::lock_guard<std::mutex> lk(g_tmu);
  TimingRec r;
  r.cls = cls;
  if (!g_pool.empty()) {
    r.a = g_pool.back().first;
    r.b = g_pool.back().second;
    g_pool.pop_back();
  } else {
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  }
  cudaEventRecord(r.a, st);
  g_recs.push_back(r);
}
void timing_end(cudaStream_t st) {
  if (!g_timing) return;
  std::lock_guard<std::mutex> lk(g_tmu);
  if (!g_recs.empty()) cudaEventRecord(g_recs.back().b, st);
}
static const char* kclass_names[KC_COUNT] = {
    "pack_weights", "node_encoder", "edge_encoder", "node_pre", "edge_step", "node_update", "decoder",
    "decoder_bwd", "node_update_bwd", "edge_step_bwd", "node_pre_bwd", "encoder_bwd", "ln_finalize", "grad_reduce",
    "loss", "loss_bwd",
    "jvp_node_encoder", "jvp_edge_encoder", "jvp_node_pre", "jvp_edge_step", "jvp_node_update", "jvp_decoder",
    "vjp_decoder", "vjp_node_update", "vjp_edge_step", "vjp_node_pre", "vjp_encoder", "vjp_ln_finalize"};
}  // namespace pdg

extern "C" long long pdg_launch_count(int reset) {
  long long v = pdg::g_launches.load();
  if (reset) pdg::g_launches = 0;
  return v;
}
extern "C" int pdg_timing_enable(int on) {
  std::lock_guard<std::mutex> lk(pdg::g_tmu);
  pdg::g_timing = on != 0;
  return 0;
}
extern "C" int pdg_timing_classes(void) { return pdg::KC_COUNT; }
extern "C" const char* pdg_timing_class_name(int cls) {
  return (cls >= 0 && cls < pdg::KC_COUNT) ? pdg::kclass_names[cls] : "";
}
// Sums the elapsed time of every recorded (begin, end) pair per class and clears the log.
// Synchronises on the recorded events (call it outside timed regions).
extern "C" int pdg_timing_collect(double* ms_per_class, long long* count_per_class) {
  std::lock_guard<std::mutex> lk(pdg::g_tmu);
  for (int i = 0; i < pdg::KC_COUNT; ++i) { ms_per_class[i] = 0; count_per_class[i] = 0; }
  for (auto& r : pdg::g_recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ms_per_class[r.cls] += ms;
      count_per_class[r.cls] += 1;
    }
    pdg::g_pool.push_back({r.a, r.b});
  }
  pdg::g_recs.clear();
  return 0;
}

extern "C" const char* pdg_last_error(void) { return pdg::g_err; }
extern "C" int pdg_version(void) { return 100; }
extern "C" int pdg_num_sms(void) { return pdg::num_sms(); }
extern "C" int pdg_persistent_grid(int n_tiles, int sms) {
  if (n_tiles <= 0 || sms <= 0) return 0;
  return pdg::balanced_grid(n_tiles, sms);
}
