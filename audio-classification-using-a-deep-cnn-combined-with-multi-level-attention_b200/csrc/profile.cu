// Launch accounting and optional per-stage CUDA-event timing (used by bench.py for the roofline line).
// Disabled by default: when off, stage marks cost one relaxed atomic load.
#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/vggish_mla_b200.h"
#include "kernels.cuh"

namespace vmb {

namespace {
std::atomic<long long> g_launches{0};
std::atomic<int> g_prof_on{0};
std::mutex g_prof_mu;
struct Span { cudaEvent_t a, b; int stage; };
std::vector<Span> g_spans;
std::vector<cudaEvent_t> g_pool;
double g_ms[VMB_NUM_STAGES];
long long g_calls[VMB_NUM_STAGES];

cudaEvent_t take_event() {
  if (!g_pool.empty()) {
    cudaEvent_t e = g_pool.back();
    g_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
}  // namespace

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

StageTimer::StageTimer(int stage, cudaStream_t st) : stage_(stage), st_(st), on_(g_prof_on.load(std::memory_order_relaxed) != 0) {
  if (!on_) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  a_ = take_event();
  b_ = take_event();
  cudaEventRecord(a_, st_);
}
StageTimer::~StageTimer() {
  if (!on_) return;
  cudaEventRecord(b_, st_);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_spans.push_back(Span{a_, b_, stage_});
}

}  // namespace vmb

extern "C" {

long long vmb_launch_count(void) { return vmb::g_launches.load(std::memory_order_relaxed); }

int vmb_profile_enable(int on) {
  vmb::g_prof_on.store(on ? 1 : 0, std::memory_order_relaxed);
  return 0;
}

int vmb_profile_collect(double* ms_per_stage, long long* calls_per_stage, int reset) {
  std::lock_guard<std::mutex> lk(vmb::g_prof_mu);
  for (auto& s : vmb::g_spans) {
    float ms = 0.f;
    if (cudaEventSynchronize(s.b) == cudaSuccess && cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess &&
        s.stage >= 0 && s.stage < VMB_NUM_STAGES) {
      vmb::g_ms[s.stage] += ms;
      vmb::g_calls[s.stage] += 1;
    }
    vmb::g_pool.push_back(s.a);
    vmb::g_pool.push_back(s.b);
  }
  vmb::g_spans.clear();
  for (int i = 0; i < VMB_NUM_STAGES; ++i) {
    if (ms_per_stage) ms_per_stage[i] = vmb::g_ms[i];
    if (calls_per_stage) calls_per_stage[i] = vmb::g_calls[i];
    if (reset) {
      vmb::g_ms[i] = 0;
      vmb::g_calls[i] = 0;
    }
  }
  return 0;
}

}  // extern "C"
