// Opt-in per-stage device timing and launch counting (diagnostics for bench.py's roofline line).
// Disabled by default: when off, no events are created and the hot path is untouched.
#pragma once
#include <cuda_runtime.h>
#include <mutex>
#include <vector>

namespace egnn {

enum Stage { STAGE_SELECT = 0, STAGE_NODE_PRE = 1, STAGE_PAIR = 2, STAGE_NODE_POST = 3, STAGE_COUNT = 4 };

struct Profiler {
  std::mutex mu;
  bool on = false;
  struct Span { cudaEvent_t a, b; int stage; };
  std::vector<Span> spans;
  long long launches = 0;
  static Profiler& get() { static Profiler p; return p; }
};

// Brackets the kernels of one stage with two events on the launch stream.
struct StageTimer {
  cudaStream_t st; int stage; cudaEvent_t a = nullptr; bool active;
  StageTimer(cudaStream_t s, int stage_) : st(s), stage(stage_) {
    Profiler& p = Profiler::get();
    active = p.on;
    if (active) { cudaEventCreate(&a); cudaEventRecord(a, st); }
  }
  ~StageTimer() {
    if (!active) return;
    cudaEvent_t b; cudaEventCreate(&b); cudaEventRecord(b, st);
    Profiler& p = Profiler::get();
    std::lock_guard<std::mutex> g(p.mu);
    p.spans.push_back({a, b, stage});
  }
};

inline void count_launch() {
  Profiler& p = Profiler::get();
  if (p.on) { std::lock_guard<std::mutex> g(p.mu); p.launches += 1; }
}

}  // namespace egnn
