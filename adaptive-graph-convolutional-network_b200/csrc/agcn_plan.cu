// Batch topology ("plan") and layout conversion between the reference's zero-padded wire layout
// (models/tf_modules/graph_topology.py:84-135) and the packed HBM layout of this library.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <numeric>

#include "agcn_internal.cuh"

namespace agcn {

static thread_local std::string t_error;
std::atomic<uint64_t> g_launches{0};

void set_error(const std::string& msg) { t_error = msg; }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  t_error = std::string(what) + " failed: " + cudaGetErrorString(e) + " (" + file + ":" + std::to_string(line) + ")";
  return (e == cudaErrorNoDevice || e == cudaErrorNoKernelImageForDevice || e == cudaErrorInsufficientDriver)
             ? AGCN_ERR_NO_DEVICE
             : AGCN_ERR_CUDA;
}

int fork_streams(const agcn_plan* plan, cudaStream_t main, int n_aux) {
  if (n_aux <= 0) return AGCN_OK;
  AGCN_CUDA(cudaEventRecord(plan->ev_fork, main));
  for (int i = 0; i < n_aux && i < 3; ++i) AGCN_CUDA(cudaStreamWaitEvent(plan->aux[i], plan->ev_fork, 0));
  return AGCN_OK;
}

int join_streams(const agcn_plan* plan, cudaStream_t main, int n_aux) {
  for (int i = 0; i < n_aux && i < 3; ++i) {
    AGCN_CUDA(cudaEventRecord(plan->ev_join[i], plan->aux[i]));
    AGCN_CUDA(cudaStreamWaitEvent(main, plan->ev_join[i], 0));
  }
  return AGCN_OK;
}

// ------------------------------------------------------------------ pack / unpack kernels
// One warp per padded row: rows < n_g are copied, rows >= n_g are written as +0.0f (unpack) or
// skipped (pack).  graphconv.py:153 (tf.slice) and :249-251 (tf.pad).
__global__ void pack_nodes_kernel(const float* __restrict__ padded, float* __restrict__ packed,
                                  const int32_t* __restrict__ n_nodes, const int32_t* __restrict__ node_off, int B,
                                  int Nmax, int F, int to_padded) {
  const int warps_per_block = blockDim.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (row >= (int64_t)B * Nmax) return;
  const int lane = threadIdx.x & 31;
  const int g = (int)(row / Nmax), i = (int)(row % Nmax);
  const int n = n_nodes[g];
  const float* pp = padded + row * F;
  float* ppw = const_cast<float*>(pp);
  if (i < n) {
    const int64_t prow = (int64_t)node_off[g] + i;
    if (to_padded) {
      for (int c = lane; c < F; c += 32) ppw[c] = packed[prow * F + c];
    } else {
      for (int c = lane; c < F; c += 32) packed[prow * F + c] = pp[c];
    }
  } else if (to_padded) {
    for (int c = lane; c < F; c += 32) ppw[c] = 0.0f;
  }
}

__global__ void pack_lap_kernel(const float* __restrict__ padded, float* __restrict__ packed,
                                const int32_t* __restrict__ n_nodes, const int64_t* __restrict__ lap_off, int B,
                                int Nmax, int to_padded) {
  const int warps_per_block = blockDim.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (row >= (int64_t)B * Nmax) return;
  const int lane = threadIdx.x & 31;
  const int g = (int)(row / Nmax), i = (int)(row % Nmax);
  const int n = n_nodes[g];
  float* ppw = const_cast<float*>(padded) + row * Nmax;
  if (i < n) {
    float* pk = packed + lap_off[g] + (int64_t)i * n;
    if (to_padded) {
      for (int c = lane; c < Nmax; c += 32) ppw[c] = (c < n) ? pk[c] : 0.0f;
    } else {
      for (int c = lane; c < n; c += 32) pk[c] = ppw[c];
    }
  } else if (to_padded) {
    for (int c = lane; c < Nmax; c += 32) ppw[c] = 0.0f;
  }
}


// Padded -> packed over the REAL rows only (the direction every training step takes).  When the padded array is a pinned
// host buffer read in place over PCIe, the kernel lives for the PCIe transfer time beside the previous training step.
// Three measurements of round 2 (tools/pack_time.py, a pack-grid sweep, tools/e2e_host_split.py) shaped it:
//  1. A zero-copy read crosses PCIe per L2 sector group: unaligned scalar row reads decay to 32-byte requests and the
//     link's outstanding-read tags saturate at ~18 GB/s whatever the number of threads; whole aligned 128-byte lines
//     (eight lanes x float4, elements outside the segment dropped) reach 40 GB/s.
//  2. What the transfer costs the step running beside it does not depend on the SMs it occupies (8 x 1024 threads and
//     148 x 32 threads cost the same) and a plain copy-engine cudaMemcpyAsync of the same bytes costs it too, while a graph
//     launch of the step is immune (tools/replay_vs_pcie.py).  The reading that fits (inferred from the timings): bulk
//     GPU-initiated PCIe reads delay the front end's fetches of the step's ~80 eager launch commands from host memory
//     (ToxCast: 0.69 ms per step alone, 0.81-0.85 ms with 8 MB arriving beside it; a feeder thread that gathers on the
//     host and sends one contiguous copy was slower still, 0.90 ms).
//  3. So the pack runs on TWO 1024-thread CTAs whatever the batch: ~130 KB of reads in flight is 28-47 GB/s, and the
//     gaps it leaves let the command fetches through.  Pipelined loop, ms per step with 2 / 4 / 8 / 14-16 CTAs:
//     ToxCast 0.81 / 0.81 / 0.85 / -, ragged clouds (C4, 42 MB) 1.62 / 1.64 / - / 2.00, ModelNet40-shape (C3, 134 MB)
//     2.86 / - / 2.94 / 3.22; one CTA is too slow (C4: 3.1 ms, transfer-bound).
__device__ __forceinline__ int graph_of_row(const int32_t* __restrict__ node_off, int B, int r) {
  int lo = 0, hi = B;   // node_off[lo] <= r < node_off[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (node_off[mid] <= r) lo = mid; else hi = mid;
  }
  return lo;
}

// The source is read in whole, aligned 128-byte lines (eight lanes x float4 per line): a zero-copy read over PCIe is
// issued per L2 sector group, and 32-byte requests (what unaligned scalar row reads decay to) saturate the link's
// outstanding-read tags at ~18 GB/s, whatever the number of threads.  Elements of a line outside the segment are dropped;
// the destination (device memory) takes scalar stores.
//   LAP = false: one segment per graph, its n real rows of X are contiguous in both layouts (n F floats); a warp per graph,
//                its four lane groups striding over the lines, PACK_U lines per group in flight;
//   LAP = true : one segment per row of L (n floats at stride Nmax); a warp takes four rows at a time, a lane group each.
constexpr int PACK_U = 4;
template <bool LAP>
__global__ void __launch_bounds__(1024) pack_lines_kernel(const float* __restrict__ padded, float* __restrict__ packed,
                                                         const int32_t* __restrict__ n_nodes,
                                                         const int32_t* __restrict__ node_off,
                                                         const int64_t* __restrict__ lap_off, int B, int Nmax, int F, int R,
                                                         int64_t total) {
  const int lane = threadIdx.x & 31, q = lane >> 3, l8 = lane & 7;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  // line `l` of a segment that starts at float s0 (first line starts at a0 = s0 rounded down to 32 floats)
  auto load_line = [&](int64_t a0, int l, bool on) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t idx = a0 + 32 * (int64_t)l + 4 * l8;
    if (on) {
      if (idx + 4 <= total) {
        v = __ldg(reinterpret_cast<const float4*>(padded + idx));
      } else {   // the last, partial float4 of the array
        if (idx < total) v.x = __ldg(padded + idx);
        if (idx + 1 < total) v.y = __ldg(padded + idx + 1);
        if (idx + 2 < total) v.z = __ldg(padded + idx + 2);
      }
    }
    return v;
  };
  auto store_line = [&](int64_t a0, int l, int64_t s0, int64_t len, int64_t d0, const float4& v, bool on) {
    if (!on) return;
    const int64_t o = a0 + 32 * (int64_t)l + 4 * l8 - s0;   // offset of v.x in the segment
    float* dst = packed + d0 + o;
    if (o >= 0 && o < len) dst[0] = v.x;
    if (o + 1 >= 0 && o + 1 < len) dst[1] = v.y;
    if (o + 2 >= 0 && o + 2 < len) dst[2] = v.z;
    if (o + 3 >= 0 && o + 3 < len) dst[3] = v.w;
  };
  if (!LAP) {
    for (int g = w; g < B; g += warps) {
      const int64_t s0 = (int64_t)g * Nmax * F, len = (int64_t)n_nodes[g] * F, d0 = (int64_t)node_off[g] * F;
      const int64_t a0 = s0 & ~(int64_t)31;
      const int nl = (int)((s0 - a0 + len + 31) >> 5);
      for (int l = q; l < nl; l += 4 * PACK_U) {
        float4 v[PACK_U];
#pragma unroll
        for (int u = 0; u < PACK_U; ++u) v[u] = load_line(a0, l + 4 * u, l + 4 * u < nl);
#pragma unroll
        for (int u = 0; u < PACK_U; ++u) store_line(a0, l + 4 * u, s0, len, d0, v[u], l + 4 * u < nl);
      }
    }
  } else {
    for (int r0 = 4 * w; r0 < R; r0 += 4 * warps) {
      const int r = r0 + q;
      int64_t s0 = 0, len = 0, d0 = 0;
      if (r < R) {
        const int g = graph_of_row(node_off, B, r);
        const int i = r - node_off[g], n = n_nodes[g];
        s0 = ((int64_t)g * Nmax + i) * Nmax;
        d0 = lap_off[g] + (int64_t)i * n;
        len = n;
      }
      const int64_t a0 = s0 & ~(int64_t)31;
      const int nl = len ? (int)((s0 - a0 + len + 31) >> 5) : 0;
      for (int l = 0; __any_sync(0xffffffffu, l < nl); l += PACK_U) {
        float4 v[PACK_U];
#pragma unroll
        for (int u = 0; u < PACK_U; ++u) v[u] = load_line(a0, l + u, l + u < nl);
#pragma unroll
        for (int u = 0; u < PACK_U; ++u) store_line(a0, l + u, s0, len, d0, v[u], l + u < nl);
      }
    }
  }
}

// fallback for a source that is not 16-byte aligned: one row per warp, scalar loads
__global__ void __launch_bounds__(1024) pack_rows_kernel(const float* __restrict__ padded, float* __restrict__ packed,
                                                        const int32_t* __restrict__ n_nodes,
                                                        const int32_t* __restrict__ node_off,
                                                        const int64_t* __restrict__ lap_off, int B, int Nmax, int F,
                                                        int R, int lap) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < R; r += warps) {
    const int g = graph_of_row(node_off, B, r);
    const int i = r - node_off[g];
    const float* __restrict__ src;
    float* __restrict__ dst;
    int len;
    if (lap) {
      const int n = n_nodes[g];
      src = padded + ((int64_t)g * Nmax + i) * Nmax;
      dst = packed + lap_off[g] + (int64_t)i * n;
      len = n;
    } else {
      src = padded + ((int64_t)g * Nmax + i) * F;
      dst = packed + (int64_t)r * F;
      len = F;
    }
    for (int c = lane; c < len; c += 32) dst[c] = __ldg(src + c);
  }
}

// grid of the pack kernels (finding 3 above)
constexpr int PACK_CTAS = 2, PACK_THREADS = 1024;
static void pack_shape(int64_t warp_items, unsigned* ctas, unsigned* threads) {
  *threads = (unsigned)PACK_THREADS;
  *ctas = (unsigned)std::max<int64_t>(
      1, std::min<int64_t>((std::max<int64_t>(1, warp_items) * 32 + PACK_THREADS - 1) / PACK_THREADS, PACK_CTAS));
}

static void launch_pack(const agcn_plan* plan, const float* padded, float* packed, int F, int lap, cudaStream_t st) {
  unsigned ctas, threads;
  if ((reinterpret_cast<uintptr_t>(padded) & 15) != 0) {
    pack_shape(plan->R, &ctas, &threads);
    pack_rows_kernel<<<ctas, threads, 0, st>>>(padded, packed, plan->d_n, plan->d_node_off, plan->d_lap_off, plan->B,
                                              plan->Nmax, F, (int)plan->R, lap);
  } else if (lap) {
    pack_shape((plan->R + 3) / 4, &ctas, &threads);
    pack_lines_kernel<true><<<ctas, threads, 0, st>>>(padded, packed, plan->d_n, plan->d_node_off, plan->d_lap_off, plan->B,
                                                     plan->Nmax, F, (int)plan->R,
                                                     (int64_t)plan->B * plan->Nmax * plan->Nmax);
  } else {
    pack_shape(plan->B, &ctas, &threads);
    pack_lines_kernel<false><<<ctas, threads, 0, st>>>(padded, packed, plan->d_n, plan->d_node_off, plan->d_lap_off, plan->B,
                                                      plan->Nmax, F, (int)plan->R, (int64_t)plan->B * plan->Nmax * F);
  }
}

// Tiles of the recurrence kernels (agcn_cheb_tile.cu): 128-row ranges of the graphs above AGCN_FUSE_MAX_N, then the small graphs
// first-fit-decreasing into 128-row tiles under the shared-memory budget of their L matrices.  `order` lists the
// graphs largest first.  gstart gets tiles + 1 entries.
static void build_fused_tiles(const std::vector<int32_t>& n, const std::vector<int32_t>& order,
                              std::vector<int32_t>* gstart, std::vector<int32_t>* entries, int* n_small_tiles) {
  const int B = (int)n.size();
  gstart->clear();
  entries->clear();
  auto push = [&](int g, int a, int b, int c) {
    entries->push_back(g); entries->push_back(a); entries->push_back(b); entries->push_back(c);
  };
  int i = 0;
  while (i < B && n[order[i]] > AGCN_FUSE_MAX_N) ++i;  // their 128-row ranges come after the small tiles
  const int n_big = i;
  struct Open { int rows, lused; std::vector<int32_t> e; };
  std::vector<Open> open;
  size_t first_open = 0;
  const int min_n = n[order[B - 1]];
  for (; i < B; ++i) {
    const int g = order[i], ng = n[g], need = ng * (ng | 1);
    size_t t = first_open;
    for (; t < open.size(); ++t)
      if (open[t].rows + ng <= 128 && open[t].lused + need <= AGCN_FUSE_LCAP) break;
    if (t == open.size()) open.push_back(Open{0, 0, {}});
    Open& o = open[t];
    o.e.push_back(g); o.e.push_back(o.rows); o.e.push_back(ng); o.e.push_back(o.lused);
    o.rows += ng;
    o.lused += need;
    while (first_open < open.size() && open[first_open].rows + min_n > 128) ++first_open;
  }
  for (const Open& o : open) {
    gstart->push_back((int32_t)(entries->size() / 4));
    entries->insert(entries->end(), o.e.begin(), o.e.end());
  }
  if (n_small_tiles) *n_small_tiles = (int)gstart->size();
  for (int b = 0; b < n_big; ++b) {
    const int g = order[b];
    for (int r = 0; r < n[g]; r += 128) {
      gstart->push_back((int32_t)(entries->size() / 4));
      push(g, r, std::min(128, n[g] - r), -1);
    }
  }
  gstart->push_back((int32_t)(entries->size() / 4));
}


// The plan tables reach the device through a kernel that reads the pinned staging buffer over PCIe (unified
// addressing), not through a copy-engine transfer: a training loop that prefetches the next batch keeps the
// host-to-device engine busy with a 100 MB copy, and a tiny cudaMemcpyAsync queued behind it would hold back the
// first kernels of the current step.
__global__ void upload_tables_kernel(const int4* __restrict__ src, int4* __restrict__ dst, size_t n16) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = src[i];
}

// Same reason for zero fills on the hot path: a kernel, never the copy engine.
__global__ void zero_fill_kernel(float* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = 0.f;
}
int zero_async(float* dst, size_t floats, cudaStream_t st) {
  if (floats == 0) return AGCN_OK;
  zero_fill_kernel<<<(unsigned)std::min<size_t>((floats + 255) / 256, 592), 256, 0, st>>>(dst, floats);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// ------------------------------------------------------------------ pooled plan resources
// A plan is created for every batch of a training loop, so creating it must not synchronise anything: the side
// streams / events come from a process-wide pool, the offset tables travel through pooled pinned staging buffers
// (reused only after the copy that read them has completed) and the device block is stream-ordered
// (cudaMallocAsync / cudaFreeAsync).
struct PlanRes {
  cudaStream_t aux[3] = {nullptr, nullptr, nullptr}, side = nullptr, big = nullptr, head = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr}, ev_side_fork = nullptr, ev_side_join = nullptr,
              ev_big_fork = nullptr, ev_big_join = nullptr, ev_head_fork = nullptr, ev_head_join = nullptr,
              ev_ready = nullptr;
  int device = -1;
};
struct Staging {
  void* host = nullptr;
  size_t bytes = 0;
  cudaEvent_t done = nullptr;
  int device = -1;
};
static std::mutex g_pool_mu;
static std::vector<PlanRes> g_res_pool;
static std::vector<Staging> g_staging_pool;

static cudaError_t acquire_res(PlanRes* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  {
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (size_t i = 0; i < g_res_pool.size(); ++i)
      if (g_res_pool[i].device == dev) {
        *out = g_res_pool[i];
        g_res_pool.erase(g_res_pool.begin() + i);
        return cudaSuccess;
      }
  }
  PlanRes r;
  r.device = dev;
  for (int i = 0; i < 3 && e == cudaSuccess; ++i) {
    e = cudaStreamCreateWithFlags(&r.aux[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_join[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r.side, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_side_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_side_join, cudaEventDisableTiming);
  // the chain of the graphs above the tiles (a handful of CTAs that each need most of an SM's shared memory) gets the
  // highest priority: its CTAs are placed before the hundreds of tile CTAs launched beside it, instead of behind them
  if (e == cudaSuccess) {
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) { lo = hi = 0; (void)cudaGetLastError(); }
    e = cudaStreamCreateWithPriority(&r.big, cudaStreamNonBlocking, hi);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_big_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_big_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r.head, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_head_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_head_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev_ready, cudaEventDisableTiming);
  *out = r;
  return e;
}

static void release_res(const PlanRes& r) {
  std::lock_guard<std::mutex> lock(g_pool_mu);
  g_res_pool.push_back(r);
}

static cudaError_t acquire_staging(size_t bytes, Staging* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  {
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (size_t i = 0; i < g_staging_pool.size(); ++i) {
      Staging& s = g_staging_pool[i];
      if (s.device != dev || s.bytes < bytes) continue;
      const cudaError_t q = cudaEventQuery(s.done);
      if (q == cudaSuccess) {
        *out = s;
        g_staging_pool.erase(g_staging_pool.begin() + i);
        return cudaSuccess;
      }
      // still being read by the upload of a plan that was destroyed early: cudaErrorNotReady is not an error and
      // must not stay in the runtime's last-error slot (the next AGCN_LAUNCH_CHECK would report it)
      (void)cudaGetLastError();
    }
  }
  Staging s;
  s.device = dev;
  s.bytes = std::max<size_t>((bytes + 65535) & ~(size_t)65535, (size_t)1 << 18);
  e = cudaMallocHost(&s.host, s.bytes);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming);
  *out = s;
  return e;
}

static void release_staging(const Staging& s) {
  if (!s.host) return;
  std::lock_guard<std::mutex> lock(g_pool_mu);
  g_staging_pool.push_back(s);
}

// Every entry point that enqueues work for a plan: order the stream after the upload of the plan's tables (when it
// is not the stream the plan was created on) and remember it, so that agcn_plan_destroy releases the device block
// in the order of the last stream that used it.
int plan_use(const agcn_plan* plan, cudaStream_t st) {
  agcn_plan* p = const_cast<agcn_plan*>(plan);
  if (!p->ready_done && st != p->create_stream) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    AGCN_CUDA(cudaStreamIsCapturing(st, &cs));
    if (cs == cudaStreamCaptureStatusNone) {  // (a plan used under capture was uploaded long before)
      const cudaError_t q = cudaEventQuery(p->ev_ready);
      if (q == cudaSuccess) {
        p->ready_done = true;
      } else {
        (void)cudaGetLastError();  // cudaErrorNotReady is not an error
        AGCN_CUDA(cudaStreamWaitEvent(st, p->ev_ready, 0));
      }
    }
  }
  p->last_stream = st;
  return AGCN_OK;
}

}  // namespace agcn

using namespace agcn;

extern "C" {

int agcn_version(void) { return 100; }
const char* agcn_last_error(void) { return t_error.c_str(); }
uint64_t agcn_launch_count(void) { return g_launches.load(); }

int agcn_plan_create(const int32_t* n_nodes_host, int32_t B, int32_t Nmax, void* stream, agcn_plan** out) {
  AGCN_REQUIRE(n_nodes_host && out, "null pointer");
  AGCN_REQUIRE(B >= 1 && Nmax >= 1, "B and Nmax must be positive");
  agcn_plan* p = new agcn_plan();
  p->B = B;
  p->Nmax = Nmax;
  p->n.assign(n_nodes_host, n_nodes_host + B);
  p->node_off.resize(B + 1);
  p->lap_off.resize(B + 1);
  p->node_off[0] = 0;
  p->lap_off[0] = 0;
  for (int g = 0; g < B; ++g) {
    const int n = p->n[g];
    if (n < 1 || n > Nmax) {
      delete p;
      set_error("invalid argument: n_nodes[g] must be in [1, Nmax]");
      return AGCN_ERR_INVALID;
    }
    p->node_off[g + 1] = p->node_off[g] + n;
    p->lap_off[g + 1] = p->lap_off[g] + (int64_t)n * n;
    p->max_n = std::max(p->max_n, n);
  }
  p->R = p->node_off[B];
  p->LL = p->lap_off[B];
  p->uniform_n = p->max_n;
  for (int g = 0; g < B; ++g)
    if (p->n[g] != p->max_n) p->uniform_n = 0;
  // largest first: long-running graphs are scheduled first (LPT)
  p->order.resize(B);
  std::iota(p->order.begin(), p->order.end(), 0);
  std::stable_sort(p->order.begin(), p->order.end(), [&](int a, int b) { return p->n[a] > p->n[b]; });
  int pos = 0;
  while (pos < B && p->n[p->order[pos]] > AGCN_SMALL_MAX) ++pos;
  p->large_count = pos;
  // Mid-size graphs (above the fused tiles, up to AGCN_SMALL_MAX): a handful per batch (molecules) run their
  // recurrences in one per-graph shared-memory kernel; when they are the bulk of the batch (the N = 128 sweep points)
  // the row-tiled products (tensor cores) are ~2x faster (profiles/r01_m_layer_sweep.jsonl).
  {
    int mid = 0;
    for (int i = pos; i < B && p->n[p->order[i]] > AGCN_FUSE_MAX_N; ++i) ++mid;
    if (mid >= AGCN_MID_TILED_MIN) p->cheb_small_max = AGCN_FUSE_MAX_N;
  }
  for (int i = 0; i < B && p->n[p->order[i]] > p->cheb_small_max; ++i) {
    const int g = p->order[i];
    if (i <= p->large_count) p->big_tile_start.push_back((int32_t)p->tile_graph.size());
    if (i == p->large_count) p->big_tiles = (int)p->tile_graph.size();
    for (int r = 0; r < p->n[g]; r += 64) {
      p->tile_graph.push_back(g);
      p->tile_row.push_back(r);
    }
  }
  p->large_tiles = (int)p->tile_graph.size();
  if ((int)p->big_tile_start.size() <= p->large_count) {  // every tiled graph is a big one
    p->big_tile_start.push_back(p->large_tiles);
    p->big_tiles = p->large_tiles;
  }
  static const int limits[] = {AGCN_SMALL_MAX, AGCN_FUSE_MAX_N, 32, 16};  // bucket = (limit_next, limit]
  for (int b = 0; b < 4 && pos < B; ++b) {
    const int lo = (b + 1 < 4) ? limits[b + 1] : 0;
    const int start = pos;
    while (pos < B && p->n[p->order[pos]] > lo) ++pos;
    if (pos > start) p->buckets.push_back(Bucket{start, pos - start, p->n[p->order[start]], limits[b]});
  }
  build_fused_tiles(p->n, p->order, &p->ft_gstart, &p->ft_entries, &p->ft_small_tiles);
  p->ft_tiles = (int)p->ft_gstart.size() - 1;
  // device block: n[B] node_off[B+1] order[B] tile_graph[T] tile_row[T] (int32) then lap_off[B+1] (int64)
  const size_t T = (size_t)p->large_tiles;
  const size_t NB = p->big_tile_start.size();
  const size_t n32 = (size_t)B + (B + 1) + B + 2 * T + NB + p->ft_gstart.size();
  const size_t off64 = (n32 * 4 + 15) / 16 * 16;
  const size_t off_ft = (off64 + (size_t)(B + 1) * 8 + 15) / 16 * 16;  // int4 entries of the fused tiles
  const size_t bytes = off_ft + p->ft_entries.size() * 8;  // device entries carry node_off / lap_off of their graph
  cudaStream_t st = (cudaStream_t)stream;
  PlanRes res;
  Staging stg;
  cudaError_t e = acquire_res(&res);
  if (e == cudaSuccess) e = acquire_staging(bytes, &stg);
  if (e != cudaSuccess) {
    int rc = cuda_fail(e, "agcn_plan_create (resources)", __FILE__, __LINE__);
    delete p;
    return rc;
  }
  char* host = reinterpret_cast<char*>(stg.host);
  std::memset(host, 0, bytes);
  int32_t* h32 = reinterpret_cast<int32_t*>(host);
  std::memcpy(h32, p->n.data(), (size_t)B * 4);
  std::memcpy(h32 + B, p->node_off.data(), (size_t)(B + 1) * 4);
  std::memcpy(h32 + 2 * B + 1, p->order.data(), (size_t)B * 4);
  if (T) {
    std::memcpy(h32 + 3 * B + 1, p->tile_graph.data(), T * 4);
    std::memcpy(h32 + 3 * B + 1 + T, p->tile_row.data(), T * 4);
  }
  std::memcpy(h32 + 3 * B + 1 + 2 * T, p->big_tile_start.data(), NB * 4);
  std::memcpy(h32 + 3 * B + 1 + 2 * T + NB, p->ft_gstart.data(), p->ft_gstart.size() * 4);
  std::memcpy(host + off64, p->lap_off.data(), (size_t)(B + 1) * 8);
  {
    int32_t* de = reinterpret_cast<int32_t*>(host + off_ft);
    for (size_t en = 0; en < p->ft_entries.size() / 4; ++en) {
      const int32_t* src = &p->ft_entries[4 * en];
      const int64_t lo = p->lap_off[src[0]];
      de[8 * en + 0] = src[0]; de[8 * en + 1] = src[1]; de[8 * en + 2] = src[2]; de[8 * en + 3] = src[3];
      de[8 * en + 4] = p->node_off[src[0]];
      de[8 * en + 5] = (int32_t)(uint32_t)(lo & 0xffffffffll);
      de[8 * en + 6] = (int32_t)(uint32_t)((uint64_t)lo >> 32);
      de[8 * en + 7] = 0;
    }
  }
  for (int i = 0; i < 3; ++i) { p->aux[i] = res.aux[i]; p->ev_join[i] = res.ev_join[i]; }
  p->ev_fork = res.ev_fork; p->side = res.side; p->ev_side_fork = res.ev_side_fork; p->ev_side_join = res.ev_side_join;
  p->big = res.big; p->ev_big_fork = res.ev_big_fork; p->ev_big_join = res.ev_big_join; p->ev_ready = res.ev_ready;
  p->head = res.head; p->ev_head_fork = res.ev_head_fork; p->ev_head_join = res.ev_head_join;
  p->res_device = res.device;
  p->staging_host = stg.host; p->staging_bytes = stg.bytes; p->staging_done = stg.done;
  p->create_stream = st;
  p->last_stream = st;
  const size_t n16 = (bytes + 15) / 16;
  e = cudaMallocAsync(&p->d_block, n16 * 16, st);
  if (e == cudaSuccess) {
    upload_tables_kernel<<<(unsigned)std::min<size_t>((n16 + 255) / 256, 64), 256, 0, st>>>(
        reinterpret_cast<const int4*>(host), reinterpret_cast<int4*>(p->d_block), n16);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaEventRecord(stg.done, st);   // the staging buffer may be reused once this has passed
  if (e == cudaSuccess) e = cudaEventRecord(p->ev_ready, st);
  if (e != cudaSuccess) {
    int rc = cuda_fail(e, "agcn_plan_create", __FILE__, __LINE__);
    agcn_plan_destroy(p);
    return rc;
  }
  int32_t* d32 = reinterpret_cast<int32_t*>(p->d_block);
  p->d_n = d32;
  p->d_node_off = d32 + B;
  p->d_order = d32 + 2 * B + 1;
  p->d_tile_graph = d32 + 3 * B + 1;
  p->d_tile_row = d32 + 3 * B + 1 + T;
  p->d_big_tile_start = d32 + 3 * B + 1 + 2 * T;
  p->d_ft_gstart = d32 + 3 * B + 1 + 2 * T + NB;
  p->d_lap_off = reinterpret_cast<int64_t*>(reinterpret_cast<char*>(p->d_block) + off64);
  p->d_ft_entries = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(p->d_block) + off_ft);
  *out = p;
  return AGCN_OK;
}

int agcn_fused_tiles_host(const int32_t* n_nodes_host, int32_t B, int32_t* gstart_out, int32_t gstart_cap,
                          int32_t* entries_out, int32_t entries_cap, int32_t* tiles_out, int32_t* n_entries_out) {
  AGCN_REQUIRE(n_nodes_host && B >= 1 && tiles_out && n_entries_out, "fused_tiles_host: bad arguments");
  std::vector<int32_t> n(n_nodes_host, n_nodes_host + B), order(B), gs, en;
  for (int g = 0; g < B; ++g) AGCN_REQUIRE(n[g] >= 1, "n_nodes[g] must be >= 1");
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return n[a] > n[b]; });
  build_fused_tiles(n, order, &gs, &en, nullptr);
  *tiles_out = (int32_t)gs.size() - 1;
  *n_entries_out = (int32_t)(en.size() / 4);
  if (gstart_out && entries_out) {
    AGCN_REQUIRE(gstart_cap >= (int32_t)gs.size() && entries_cap >= (int32_t)en.size(), "fused_tiles_host: buffers too small");
    std::memcpy(gstart_out, gs.data(), gs.size() * 4);
    std::memcpy(entries_out, en.data(), en.size() * 4);
  }
  return AGCN_OK;
}

int agcn_plan_destroy(agcn_plan* p) {
  if (!p) return AGCN_OK;
  // stream-ordered: nothing is synchronised; the block is released after the last work queued for this plan
  if (p->d_block) cudaFreeAsync(p->d_block, p->last_stream);
  if (p->ev_ready) {
    PlanRes r;
    for (int i = 0; i < 3; ++i) { r.aux[i] = p->aux[i]; r.ev_join[i] = p->ev_join[i]; }
    r.ev_fork = p->ev_fork; r.side = p->side; r.ev_side_fork = p->ev_side_fork; r.ev_side_join = p->ev_side_join;
    r.big = p->big; r.ev_big_fork = p->ev_big_fork; r.ev_big_join = p->ev_big_join; r.ev_ready = p->ev_ready;
    r.head = p->head; r.ev_head_fork = p->ev_head_fork; r.ev_head_join = p->ev_head_join;
    r.device = p->res_device;
    release_res(r);
  }
  if (p->staging_host) {
    Staging sg;
    sg.host = p->staging_host; sg.bytes = p->staging_bytes; sg.done = p->staging_done; sg.device = p->res_device;
    release_staging(sg);
  }
  delete p;
  return AGCN_OK;
}

int64_t agcn_plan_total_nodes(const agcn_plan* p) { return p ? p->R : -1; }
int64_t agcn_plan_total_lap(const agcn_plan* p) { return p ? p->LL : -1; }
const int32_t* agcn_plan_node_off_host(const agcn_plan* p) { return p ? p->node_off.data() : nullptr; }
const int64_t* agcn_plan_lap_off_host(const agcn_plan* p) { return p ? p->lap_off.data() : nullptr; }

static int pack_nodes_impl(const agcn_plan* plan, const float* padded, float* packed, int32_t F, void* stream,
                           int to_padded) {
  AGCN_REQUIRE(plan && padded && packed && F >= 1, "null pointer or F < 1");
  if (int rc = plan_use(plan, (cudaStream_t)stream)) return rc;
  if (!to_padded) {
    launch_pack(plan, padded, packed, F, 0, (cudaStream_t)stream);
    AGCN_LAUNCH_CHECK();
    return AGCN_OK;
  }
  const int64_t rows = (int64_t)plan->B * plan->Nmax;
  const int wpb = 8;
  pack_nodes_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(
      padded, packed, plan->d_n, plan->d_node_off, plan->B, plan->Nmax, F, to_padded);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int agcn_pack_nodes(const agcn_plan* plan, const float* d_padded, float* d_packed, int32_t F, void* stream) {
  return pack_nodes_impl(plan, d_padded, d_packed, F, stream, 0);
}
int agcn_unpack_nodes(const agcn_plan* plan, const float* d_packed, float* d_padded, int32_t F, void* stream) {
  return pack_nodes_impl(plan, d_padded, const_cast<float*>(d_packed), F, stream, 1);
}

static int pack_lap_impl(const agcn_plan* plan, const float* padded, float* packed, void* stream, int to_padded) {
  AGCN_REQUIRE(plan && padded && packed, "null pointer");
  if (int rc = plan_use(plan, (cudaStream_t)stream)) return rc;
  if (!to_padded) {
    launch_pack(plan, padded, packed, 0, 1, (cudaStream_t)stream);
    AGCN_LAUNCH_CHECK();
    return AGCN_OK;
  }
  const int64_t rows = (int64_t)plan->B * plan->Nmax;
  const int wpb = 8;
  pack_lap_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(
      padded, packed, plan->d_n, plan->d_lap_off, plan->B, plan->Nmax, to_padded);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int agcn_pack_lap(const agcn_plan* plan, const float* d_padded, float* d_packed, void* stream) {
  return pack_lap_impl(plan, d_padded, d_packed, stream, 0);
}
int agcn_unpack_lap(const agcn_plan* plan, const float* d_packed, float* d_padded, void* stream) {
  return pack_lap_impl(plan, d_padded, const_cast<float*>(d_packed), stream, 1);
}

}  // extern "C"
