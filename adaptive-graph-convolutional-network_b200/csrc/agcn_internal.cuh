// Internal declarations shared by the translation units of libagcn_sm100.so.
// Public ABI: include/agcn_sgcll.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <vector>

#include "agcn_sgcll.h"

// Largest graph handled by the one-CTA-per-(graph, feature chunk) shared-memory kernels; bigger
// graphs go through the row-tiled kernels (agcn_graph_large.cu).
#define AGCN_SMALL_MAX 144
// Graphs above this size run their Chebyshev recurrences as row-tiled grouped GEMMs (one launch per step,
// several CTAs per graph) instead of one CTA per (graph, feature chunk).
#define AGCN_CHEB_SMALL_MAX 144
// Recurrence tiles (agcn_cheb_tile.cu): graphs up to this size are packed into 128-row tiles (whole graphs, first-fit
// decreasing) and run their Chebyshev recurrences one CTA per (tile, feature chunks); AGCN_FUSE_LCAP floats of shared
// memory hold the per-graph matrices of one tile (row pitch n | 1; two 64-node graphs fit).  Graphs between this size
// and AGCN_SMALL_MAX take one CTA row range each (the same kernel, 160 rows).
#define AGCN_FUSE_MAX_N 64
#define AGCN_FUSE_LCAP 8320
// Batches with at least this many graphs between AGCN_FUSE_MAX_N and AGCN_SMALL_MAX nodes send them through the
// row-tiled products instead of the per-graph shared-memory recurrence kernels.
#define AGCN_MID_TILED_MIN 32
// Paper-mode degree floor: a node whose similarity column sum d = sum_i exp(-dist_ij) is below 2^-80 (every other node
// farther than ~55 in the learned metric) counts as isolated, d^-1/2 := 0.  The reference adds a denormal epsilon
// (graphconv.py:196, 1.4e-45, zero under FTZ: SURVEY Q8) and then evaluates d^-1/2 ~ 1e22 on sums of denormals; the
// floor keeps d^-1/2 <= 1.1e12 and its derivative (-1/2 d^-3/2) finite in fp32.  The oracle uses the same floor.
#define AGCN_DEGREE_FLOOR 8.271806125530277e-25f

namespace agcn {

// 3xTF32 operand split: x = hi + lo (+ a remainder below 2^-23 |x|), both halves exact TF32 values.  ROUND-TO-NEAREST
// (cvt.rna) on both halves: truncation drops up to 3 * 2^-23 |x| and always in the same direction, a bias that
// accumulates linearly over a contraction; rounding leaves at most 2^-23 |x|, zero-mean (measured on the 4-layer
// network gradients: 2-3e-4 relative error with truncation against 3e-5 for plain fp32 arithmetic).
#ifdef __CUDACC__
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// Wait on an mbarrier phase (shared-space address).  A protocol bug becomes a trap instead of a hang, but only after
// TEN SECONDS of wall time on the global timer: a spin COUNT is not a time (a box whose first nvidia-smi start or
// clock ramp stalls the device for a few hundred milliseconds made a 2^24-spin limit fire in a correct kernel).
__device__ __forceinline__ void mbar_wait_shared(uint32_t addr, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  unsigned long long t0 = 0;
  while (true) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) break;
    if ((++spins & 0xFFFFu) == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 10000000000ull) __trap();
    }
  }
}
#endif

struct Bucket {
  int start;  // first index into plan->order
  int count;  // graphs in the bucket
  int max_n;  // largest n in the bucket
  int limit;  // upper size limit of the bucket (every graph of the bucket has n <= limit)
};

// A/B tuning switches (AGCN_DISABLE_TCGEN05, AGCN_DISABLE_FUSED, AGCN_BIG_TC, AGCN_CHEB_SMALL_MAX) exist only in builds
// made with -DAGCN_AB_SWITCHES (tools/gpu_check.sh); the shipped library has ONE code path per shape and reads no
// environment variables.
#ifdef AGCN_AB_SWITCHES
#include <cstdlib>
inline const char* ab_env(const char* name) { return getenv(name); }
#else
inline const char* ab_env(const char*) { return nullptr; }
#endif

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
extern std::atomic<uint64_t> g_launches;

#define AGCN_CUDA(call)                                                        \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess) return agcn::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

#define AGCN_LAUNCH_CHECK()                                                    \
  do {                                                                         \
    agcn::g_launches.fetch_add(1, std::memory_order_relaxed);                  \
    cudaError_t e__ = cudaGetLastError();                                      \
    if (e__ != cudaSuccess) return agcn::cuda_fail(e__, "kernel launch", __FILE__, __LINE__); \
  } while (0)

#define AGCN_REQUIRE(cond, msg)                                                \
  do {                                                                         \
    if (!(cond)) {                                                             \
      agcn::set_error(std::string("invalid argument: ") + msg);               \
      return AGCN_ERR_INVALID;                                                 \
    }                                                                          \
  } while (0)

}  // namespace agcn

struct agcn_plan {
  int32_t B = 0, Nmax = 0, max_n = 0;
  int32_t uniform_n = 0;   // n when every graph of the batch has the same size (then node_off[g] = g n, lap_off[g] = g n^2), else 0
  int32_t cheb_small_max = AGCN_CHEB_SMALL_MAX;  // overridable with the environment variable of the same name
  int64_t R = 0;   // total nodes
  int64_t LL = 0;  // total n^2
  std::vector<int32_t> n, node_off, order;
  std::vector<int64_t> lap_off;
  std::vector<agcn::Bucket> buckets;  // graphs with n <= AGCN_SMALL_MAX, biggest bucket first
  int large_count = 0;                // graphs with n > AGCN_SMALL_MAX are order[0 .. large_count)
  // row tiles of the graphs with n > AGCN_CHEB_SMALL_MAX: tile t covers rows [tile_row[t], tile_row[t]+64) of
  // graph tile_graph[t]
  std::vector<int32_t> tile_graph, tile_row;
  int large_tiles = 0;
  // graphs with n > AGCN_SMALL_MAX ("big": their n x n matrices never fit in shared memory) own the first
  // big_tiles entries of the tile list; big_tile_start[i] .. big_tile_start[i+1] are the tiles of order[i]
  int big_tiles = 0;
  std::vector<int32_t> big_tile_start;
  // device copies (one allocation)
  void* d_block = nullptr;
  int32_t* d_n = nullptr;
  int32_t* d_node_off = nullptr;
  int32_t* d_order = nullptr;
  int64_t* d_lap_off = nullptr;
  int32_t* d_tile_graph = nullptr;
  int32_t* d_tile_row = nullptr;
  int32_t* d_big_tile_start = nullptr;
  // fused tiles: tile t owns entries ft_gstart[t] .. ft_gstart[t+1]; an entry is {graph, first tile row, n,
  // float offset of the graph's matrix in the tile's shared-memory L region} for whole small graphs or
  // {graph, first graph row, rows, -1} for a 128-row range of a graph with n > AGCN_FUSE_MAX_N
  int ft_tiles = 0;
  int ft_small_tiles = 0;  // tiles [0, ft_small_tiles) hold whole small graphs, the rest are 128-row ranges of big ones
  std::vector<int32_t> ft_gstart, ft_entries;
  int32_t* d_ft_gstart = nullptr;
  int32_t* d_ft_entries = nullptr;  // 2 x int4 per entry: {g, r0, n, lbase} {node_off, lap_off lo, hi, 0}
  // side streams so the per-bucket launches of one phase overlap on the device
  cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr;
  cudaEvent_t ev_join[3] = {nullptr, nullptr, nullptr};
  // a fourth side stream for the parameter-gradient contraction of the backward pass (dW = T^T dY), which
  // only depends on dY and overlaps with the dX chain
  cudaStream_t side = nullptr;
  cudaEvent_t ev_side_fork = nullptr, ev_side_join = nullptr;
  // a stream for the chain of the graphs above AGCN_FUSE_MAX_N (per-graph recurrences + their tile launch), which
  // runs beside the fused launch of the small-graph tiles
  cudaStream_t big = nullptr;
  cudaEvent_t ev_big_fork = nullptr, ev_big_join = nullptr;
  // life cycle (agcn_plan.cu): streams / events / staging come from process-wide pools, the device block is
  // stream-ordered; ev_ready marks the upload of the tables on create_stream
  cudaEvent_t ev_ready = nullptr;
  cudaStream_t create_stream = nullptr, last_stream = nullptr;
  bool ready_done = false;
  int res_device = -1;
  void* staging_host = nullptr;
  size_t staging_bytes = 0;
  cudaEvent_t staging_done = nullptr;
};

namespace agcn {

// ---------------------------------------------------------------- node-level GEMMs (agcn_node_gemm.cu)
// C_z[M,N] (+)= act( sum_{s<S} A_s[M,Kd] * op(B_{z*? + s}) + bias ),   op(B) = B or B^T
struct GemmArgs {
  int M = 0, N = 0, Kd = 0;
  int S = 1;  // inner slices summed into one output
  int Z = 1;  // independent output slices (grid.z)
  const float* A0 = nullptr;  // inner slice 0
  int lda0 = 0;
  const float* A1 = nullptr;  // inner slice s >= 1: A1 + (s-1)*sliceA1
  int lda1 = 0;
  int64_t sliceA1 = 0;
  const float* B = nullptr;  // slice (z*S + s): B + (z*S+s)*sliceB
  int ldb = 0;
  int64_t sliceB = 0;
  int transB = 0;  // 0: B is [Kd,N] row-major; 1: B is [N,Kd] row-major (C = A * B^T)
  float* C = nullptr;  // output slice z: C + z*sliceC
  int ldc = 0;
  int64_t sliceC = 0;
  const float* bias = nullptr;
  const float* scale = nullptr;  // optional device scalar: the product is multiplied by scale[0] before bias / accumulate
  int act = AGCN_ACT_LINEAR;
  int accumulate = 0;  // C += result
  // tensor-core kernel only: fused loss epilogue, weighted sigmoid cross-entropy unless l2 is set (C = d loss / d logits,
  // see agcn_head.cu);
  // bce_y / bce_w are laid out like C, loss_part holds tc_gemm_loss_parts() floats
  const float* bce_y = nullptr;
  const float* bce_w = nullptr;
  int bce_ld = 0;  // row pitch of bce_y / bce_w (0: same as ldc)
  float bce_scale = 1.f;
  float* loss_part = nullptr;
  // tensor-core kernel only: prediction epilogue of the multitask head (agcn_head_predict): C receives the two-class
  // softmax of every column pair (2t, 2t+1); with bce_y set, loss_part receives the same partial sums as above
  int prob = 0;
  // tensor-core kernel only: the loss of the epilogues above is the weighted L2 of the regression head instead of the
  // sigmoid cross-entropy (loss term (w (x - y))^2, C = 2 w^2 (x - y) bce_scale; with prob set C receives x itself)
  int l2 = 0;
  // tensor-core kernel only: scratch of 8 * M * N floats; when given, long contractions with few output tiles are
  // split along K (plain outputs only: no bias / activation / accumulate / loss epilogue, ldc == N, Z == 1)
  float* split_k_partial = nullptr;
};
int tc_gemm_loss_parts(const GemmArgs& a);  // number of partial loss sums tc_gemm writes
int gemm_rows(const GemmArgs& a, cudaStream_t st);
// tcgen05 (3xTF32) implementation of the same contraction for TMA-compatible shapes (agcn_tc_gemm.cu)
bool tc_gemm_supported(const GemmArgs& a);
size_t tc_gemm_scratch_floats(int N, int Kd, int S, int Z);
int tc_gemm_split_b(const GemmArgs& a, float* scratch, cudaStream_t st);
int tc_gemm(const GemmArgs& a, const float* scratch, cudaStream_t st);

// out[(f*S + s)*N + c] = sum_r A_s[r, f] * D[r, c]     (A_s as in GemmArgs; contraction over the M rows)
struct GemmTNArgs {
  int M = 0;   // rows contracted
  int Kd = 0;  // columns of A_s  (rows of the result per slice)
  int N = 0;   // columns of D
  int S = 1;
  const float* A0 = nullptr;
  int lda0 = 0;
  const float* A1 = nullptr;
  int lda1 = 0;
  int64_t sliceA1 = 0;
  const float* D = nullptr;
  int ldd = 0;
  float* out = nullptr;  // [Kd*S, N] with row index f*S + s  (the reference's weight layout)
  float* partial = nullptr;  // scratch, gemm_tn_partial_floats() floats
};
size_t gemm_tn_partial_floats(int M, int Kd, int N, int S);
int gemm_tn(const GemmTNArgs& a, cudaStream_t st);
// tcgen05 (3xTF32, MN-major operands) implementation of the same contraction (agcn_tc_gemm.cu)
bool tc_gemm_tn_supported(const GemmTNArgs& a);
size_t tc_gemm_tn_partial_floats(const GemmTNArgs& a);
int tc_gemm_tn(const GemmTNArgs& a, cudaStream_t st);

// dYp = dY * act'(Y) (relu mask), colsum(dYp) -> dbias.  partial: act_bwd_partial_floats() floats.
size_t act_bwd_partial_floats(int64_t R, int Fo);
int act_bwd_partials(const float* dY, const float* Y, float* dYp, float* partial, int64_t R, int Fo, int act,
                     cudaStream_t st);
int act_bwd_reduce(const float* partial, float* dbias, int64_t R, int Fo, cudaStream_t st);

// ---------------------------------------------------------------- per-graph kernels (agcn_graph_small.cu)
struct GraphArgs {
  const agcn_plan* plan = nullptr;
  int F = 0, K = 0;
  int variant = 0, lap_mode = 0, metric_full = 0;
  // forward inputs
  const float* X = nullptr;      // [R,F]
  const float* XW = nullptr;     // [R,F]   X * M_L (needed when the similarity matrix is needed)
  const float* Lint = nullptr;   // packed
  const float* Lprev = nullptr;  // packed or null
  const float* alpha = nullptr;
  const float* beta = nullptr;
  // forward outputs / saved
  float* T = nullptr;       // [K-1][R][F]  Chebyshev terms T_1..T_{K-1}
  float* Lall = nullptr;    // packed L_all (null in the literal SGC_LL shortcut: L_all = I + Lint)
  float* Lall_out = nullptr;  // optional second copy of L_all (user output)
  float* resL = nullptr;    // optional output
  float* resW = nullptr;    // optional output
  float* dist = nullptr;    // packed pairwise distances (saved, paper mode)
  float* dis = nullptr;     // [R] D^-1/2 (saved, paper mode)
  float* stats = nullptr;   // [B][4]: s1, s2, sum R^2, sum Z^2 (saved)
  // backward
  const float* G = nullptr;      // [K][R][F]  dY * W_k^T
  const float* dLall_in = nullptr;
  float* dX = nullptr;           // [R,F]
  float* dL = nullptr;           // packed scratch: dL_all, as dl_parts partial sums dl_stride elements apart (the
  int dl_parts = 1;              //   recurrences of the graphs up to AGCN_SMALL_MAX nodes split the feature chunks over
  int64_t dl_stride = 0;         //   dl_parts CTAs per graph; bigger graphs use part 0 only)
  float* dLprev = nullptr;       // packed out
  float* dXW = nullptr;          // [R,F] out (metric_full)
  float* dalpha_part = nullptr;  // [B]
  float* dbeta_part = nullptr;   // [B]
  float* big_work = nullptr;     // scratch of the big-graph sweeps (big_work_floats() floats)
};
bool literal_shortcut(int variant, int lap_mode);  // L_all == I + Lint, nothing to build
int graph_build_laplacian(const GraphArgs& a, bool need_W, cudaStream_t st);
// above_n: only the graphs with more than above_n nodes (the fused tile kernels own the others)
int graph_chebyshev_fwd(const GraphArgs& a, cudaStream_t st, int above_n = 0);
int graph_recurrence_bwd(const GraphArgs& a, bool need_dL, cudaStream_t st, int above_n = 0);
int graph_laplacian_bwd(const GraphArgs& a, cudaStream_t st);
int reduce_scalar_parts(const float* parts, int B, float* out, cudaStream_t st);
// graphs with more than AGCN_SMALL_MAX nodes (agcn_graph_large.cu)
int large_chebyshev_fwd(const GraphArgs& a, cudaStream_t st);
int large_recurrence_bwd(const GraphArgs& a, float* G, bool big_only, cudaStream_t st);
// Laplacian construction / gradient for graphs with more than AGCN_SMALL_MAX nodes (agcn_graph_big.cu)
size_t big_work_floats(const agcn_plan* plan, bool full);
int big_build_laplacian(const GraphArgs& a, bool need_W, float* big_work, cudaStream_t st);
int big_dL(const GraphArgs& a, const float* U, cudaStream_t st);
int big_laplacian_bwd(const GraphArgs& a, float* big_work, cudaStream_t st);

// ---------------------------------------------------------------- row-tiled products of the graphs above
// cheb_small_max nodes (agcn_graph_large.cu, agcn_big_tc.cu):
//     Out = cmul * op(L_g) * In  (+ Add)  (- Sub)  (+ RowScale .* ScaleIn),   op(L) = L (+ I) | L^T (+ I)
// over (graph, 64-row tile) work items of the plan's tile list.
struct GroupedArgs {
  const int32_t* n_nodes;
  const int32_t* node_off;
  const int64_t* lap_off;
  const int32_t* tile_graph;
  const int32_t* tile_row;
  const float* L;
  int add_identity, transL;
  const float* In;
  const float* Sub;
  const float* Add;
  float* Out;
  float* Out2;
  float cmul;
  int F;
  const float* RowScale;  // optional: Out += RowScale[row] * ScaleIn[row, c]
  const float* ScaleIn;
  unsigned long long* dbg;  // tuning aid: timeline of the first CTA of grouped_tc_kernel (NULL in production)
  int force_uniform;        // tests: take bt::grouped_tcu_kernel whenever the batch is eligible, whatever the grid size
};
int grouped_launch(const agcn_plan* plan, int tiles, const GroupedArgs& g, cudaStream_t st);
int grouped_simt(int tiles, const GroupedArgs& g, cudaStream_t st);
// tcgen05 3xTF32 implementation (F % 4 == 0, F >= 16, 16-byte aligned node matrices)
bool grouped_tc_supported(const GroupedArgs& g);
int grouped_tc(const agcn_plan* plan, int tiles, const GroupedArgs& g, cudaStream_t st);
// pair matrices (similarity / dL) of big equal-size graphs on the tensor cores (agcn_big_tc.cu, pair_tcu_kernel)
bool pair_tc_supported(const agcn_plan* plan, int F);
int pair_tc_similarity(const agcn_plan* plan, const float* XW, int F, float* norms, float* dist, float* resW, float* rowpart,
                       int ncb, cudaStream_t st);
int pair_tc_dL(const agcn_plan* plan, const float* U, const float* X, const float* T, int F, int K, const float* dL_in,
               float* dL, cudaStream_t st);
// streaming implementation for F <= 8 (HBM-bound: the Laplacian is read once, coalesced)
bool grouped_thin_supported(const GroupedArgs& g);
int grouped_thin(int tiles, const GroupedArgs& g, cudaStream_t st);

// ---------------------------------------------------------------- tile path of a layer: parameter operands and shape
// rules (agcn_layer_operands.cu); recurrences in agcn_cheb_tile.cu, contraction in agcn_pre_tile.cu
void fused_profile_enable(int on);
int fused_profile_read(float* ms_sum, int* launches);
void prof_enable(int on);
void fused_debug_set(void* d_buf);  // per-CTA timeline buffer [CTAs][128] uint64 of the NEXT contraction / recurrence launches, or NULL
bool fused_fwd_supported(const agcn_plan* plan, int F, int Fo, int K);
bool fused_bwd_supported(const agcn_plan* plan, int F, int Fo, int K);
size_t fused_w_floats(int Nv, int Kv, int Z);  // floats of one pre-split parameter operand
int fused_fwd_prep(const float* weight, int F, int Fo, int K, float* scratch, cudaStream_t st);
int fused_bwd_prep(const float* weight, int F, int Fo, int K, float* scratch, cudaStream_t st);

// ---------------------------------------------------------------- transform product of the 128-row ranges of graphs
// above AGCN_FUSE_MAX_N (agcn_pre_tile.cu); same parameter operands as the fused tile kernels
int pre_forward(const agcn_plan* plan, int tile0, int ntiles, const float* X, const float* T, const float* wsplit,
                const float* bias, int act, int F, int Fo, int K, float* Y, cudaStream_t st);
int pre_backward(const agcn_plan* plan, int tile0, int ntiles, const float* dY, const float* Y, const float* wsplit, int F,
                 int Fo, int K, float* G, cudaStream_t st);

// ---------------------------------------------------------------- CUDA-core Chebyshev recurrences of the graphs up to
// AGCN_SMALL_MAX nodes (agcn_cheb_tile.cu): small-graph tiles on st_small, mid-size graphs on st_mid
bool cheb_tiles_has_mid(const agcn_plan* plan);
// transL: the recurrences of L^T (backward pass: V_k = T_k(L^T) dYpre)
int cheb_tiles_forward(const agcn_plan* plan, const float* X, const float* L, int add_identity, int F, int K, float* T,
                       cudaStream_t st_small, cudaStream_t st_mid, int transL = 0);
int cheb_tiles_backward(const agcn_plan* plan, const float* G, const float* L, int add_identity, int F, int K, float* dX,
                        cudaStream_t st_small, cudaStream_t st_mid);

// ---------------------------------------------------------------- live per-kernel timing (agcn_profile.cu)
// RAII bracket around ONE kernel launch in a host wrapper; records only while agcn_profile_enable(1) is in effect and
// the stream is not capturing.
class ProfScope {
 public:
  ProfScope(const char* name, cudaStream_t st);
  ~ProfScope();
  ProfScope(const ProfScope&) = delete;
  ProfScope& operator=(const ProfScope&) = delete;

 private:
  const char* name_;
  cudaStream_t st_;
  cudaEvent_t e0_;
};

// ---------------------------------------------------------------- helpers
// Bump allocator of every workspace layout: each area starts at a multiple of 256 bytes from the base.  With a null
// base every area is nullptr and `bytes` ends as what the same sequence of areas needs, so a *_workspace_bytes function
// runs the carve of its call.
struct Arena {
  char* base;
  size_t bytes = 0;
  explicit Arena(void* p) : base(static_cast<char*>(p)) {}
  void* area(size_t n) {
    void* r = base ? base + bytes : nullptr;
    bytes += (n + 255) & ~(size_t)255;
    return r;
  }
  template <typename T = float>
  T* take(size_t count) { return static_cast<T*>(area(count * sizeof(T))); }
};

int zero_async(float* dst, size_t floats, cudaStream_t st);  // zero fill by a kernel (never the copy engine)
int plan_use(const agcn_plan* plan, cudaStream_t st);  // call first in every entry point that enqueues work
int fork_streams(const agcn_plan* plan, cudaStream_t main, int n_aux);
int join_streams(const agcn_plan* plan, cudaStream_t main, int n_aux);

}  // namespace agcn
