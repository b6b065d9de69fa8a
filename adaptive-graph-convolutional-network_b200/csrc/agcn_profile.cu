// Live per-kernel timing for bench.py's roofline table: while enabled, the host wrappers of the main kernels bracket
// their launch with CUDA events on the launching stream (ProfScope); agcn_profile_read waits for them and returns
// launches and summed milliseconds per kernel name.  Off in production and never active under stream capture.
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "agcn_internal.cuh"

namespace agcn {

std::atomic<int> g_prof_on{0};

namespace {
struct ProfRec {
  const char* name;
  cudaEvent_t e0, e1;
};
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
}  // namespace

ProfScope::ProfScope(const char* name, cudaStream_t st) : name_(name), st_(st), e0_(nullptr) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    (void)cudaGetLastError();
    return;
  }
  if (cudaEventCreate(&e0_) != cudaSuccess) {
    e0_ = nullptr;
    return;
  }
  cudaEventRecord(e0_, st);
}

ProfScope::~ProfScope() {
  if (!e0_) return;
  cudaEvent_t e1 = nullptr;
  if (cudaEventCreate(&e1) != cudaSuccess) {
    cudaEventDestroy(e0_);
    return;
  }
  cudaEventRecord(e1, st_);
  std::lock_guard<std::mutex> lock(g_prof_mu);
  g_prof_recs.push_back(ProfRec{name_, e0_, e1});
}

void prof_enable(int on) { g_prof_on.store(on ? 1 : 0); }

// Drains the pending records into a per-kernel table and, if asked, a launch timeline.
int prof_drain(std::string* table, std::string* timeline = nullptr) {
  std::vector<ProfRec> recs;
  {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    recs.swap(g_prof_recs);
  }
  std::map<std::string, std::pair<int, double>> agg;
  if (timeline) timeline->clear();
  for (ProfRec& r : recs) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(r.e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.e0, r.e1);
    if (e == cudaSuccess && timeline) {   // start / end relative to the first record's start (events of any stream compare)
      float t0 = 0.f;
      e = cudaEventSynchronize(recs[0].e0);
      if (e == cudaSuccess) e = cudaEventElapsedTime(&t0, recs[0].e0, r.e0);
      *timeline += std::string(r.name) + "\t" + std::to_string(t0) + "\t" + std::to_string(t0 + ms) + "\n";
    }
    if (e != cudaSuccess) {
      for (ProfRec& d : recs) { cudaEventDestroy(d.e0); cudaEventDestroy(d.e1); }
      return cuda_fail(e, "profile read", __FILE__, __LINE__);
    }
    auto& a = agg[r.name];
    a.first += 1;
    a.second += ms;
  }
  for (ProfRec& d : recs) { cudaEventDestroy(d.e0); cudaEventDestroy(d.e1); }
  if (table) {
    table->clear();
    for (auto& kv : agg) *table += kv.first + "\t" + std::to_string(kv.second.first) + "\t" + std::to_string(kv.second.second) + "\n";
  }
  return AGCN_OK;
}

// fp32 FMA peak probe: 8 independent FMA chains per thread, `iters` trips, 2 flop per FMA
__global__ void __launch_bounds__(256) fma_probe_kernel(float* __restrict__ sink, int iters) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f,
        a7 = a0 + 7.f;
  const float b = 1.000001f, c = 1e-7f;
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
    a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
  }
  sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

}  // namespace agcn

extern "C" {

int agcn_profile_enable(int enable) {
  agcn::prof_enable(enable);
  return AGCN_OK;
}

int agcn_probe_fp32_fma(float* d_sink, int32_t iters, void* stream) {
  AGCN_REQUIRE(d_sink && iters >= 1, "probe_fp32_fma: bad arguments");
  agcn::fma_probe_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_sink, iters);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int agcn_profile_timeline(char* buf, size_t cap, size_t* needed) {
  std::string table, timeline;
  int rc = agcn::prof_drain(&table, &timeline);
  if (rc) return rc;
  if (needed) *needed = timeline.size() + 1;
  if (buf && cap) {
    const size_t n = timeline.size() < cap - 1 ? timeline.size() : cap - 1;
    timeline.copy(buf, n);
    buf[n] = 0;
  }
  return AGCN_OK;
}

int agcn_profile_read(char* buf, size_t cap, size_t* needed) {
  std::string table;
  int rc = agcn::prof_drain(&table);
  if (rc) return rc;
  if (needed) *needed = table.size() + 1;
  if (buf && cap) {
    const size_t n = table.size() < cap - 1 ? table.size() : cap - 1;
    table.copy(buf, n);
    buf[n] = 0;
  }
  return AGCN_OK;
}

}  // extern "C"
