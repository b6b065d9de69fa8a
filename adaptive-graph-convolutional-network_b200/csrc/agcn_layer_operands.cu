// Parameter operands and shape rules of the tile path of one SGC-LL layer (graphconv.py:221-247 and its reverse mode):
//
//   recurrences   agcn_cheb_tile.cu   CUDA cores, graphs up to AGCN_SMALL_MAX nodes (bigger ones: agcn_big_tc.cu)
//   contraction   agcn_pre_tile.cu    tensor cores, every packed row:  Y = act(sum_k T_k W_k + b),  G_z = dYpre W_z^T
//
// This file holds what both directions share: the hi / lo TF32 split of the weight matrix into the K-major tiles the
// contraction streams with TMA, and the predicates that say when a layer takes this path.  (Round 1 / early round 2 ran
// recurrence and contraction FUSED in one 222 KB CTA per SM here; profiles/r02f_* and DESIGN.md section 3 record why that
// design was retired: 26 us of serial worker chain against 6 us of tensor-core work per tile.)
#include <algorithm>

#include "agcn_internal.cuh"

namespace agcn {
namespace ft {

// ------------------------------------------------------------------------------------------------
// W prep: out_{hi,lo}[(z * N + n) * Kp + k] = split(W[n * sn + k * sk + z * sz])  (zero outside n < Nv, k < Kv)
// ------------------------------------------------------------------------------------------------
__global__ void prep_w_kernel(const float* __restrict__ W, long long sn, long long sk, long long sz, int Nv, int Kv,
                              int N, int Kp, int Z, float* __restrict__ hi, float* __restrict__ lo) {
  const long long total = (long long)Z * N * Kp;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(e % Kp);
    const long long rr = e / Kp;
    const int n = (int)(rr % N), z = (int)(rr / N);
    float x = 0.f;
    if (n < Nv && k < Kv) x = W[n * sn + k * sk + z * sz];
    const float h = tf32_rn(x);
    hi[e] = h;
    lo[e] = tf32_rn(x - h);
  }
}

static int pad16(int x) { return (x + 15) & ~15; }
static int pad32(int x) { return (x + 31) & ~31; }

}  // namespace ft

// ------------------------------------------------------------------------------------------------
// host API
// ------------------------------------------------------------------------------------------------
// forward: one accumulator of pad16(Fo) <= 128 columns
bool fused_fwd_supported(const agcn_plan* plan, int F, int Fo, int K) {
  return plan->ft_tiles > 0 && K >= 2 && Fo >= 1 && Fo <= 128 && F >= 1;
}

// backward: K accumulators of pad16(F) columns within the 512 TMEM columns
bool fused_bwd_supported(const agcn_plan* plan, int F, int Fo, int K) {
  if (plan->ft_tiles <= 0 || K < 2 || F > 128) return false;
  const int N = ft::pad16(F), stride = N <= 32 ? 32 : (N <= 64 ? 64 : 128);
  return K * stride <= 512;
}

size_t fused_w_floats(int Nv, int Kv, int Z) { return 2 * (size_t)Z * ft::pad16(Nv) * ft::pad32(Kv); }

// forward operand: B_s[n, k] = weight[(k*K + s)*Fo + n]  (n < Fo output columns, k < F)
int fused_fwd_prep(const float* weight, int F, int Fo, int K, float* scratch, cudaStream_t st) {
  const int N = ft::pad16(Fo), Kp = ft::pad32(F);
  const long long total = (long long)K * N * Kp;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 1184);
  ft::prep_w_kernel<<<blocks, 256, 0, st>>>(weight, 1, (long long)K * Fo, Fo, Fo, F, N, Kp, K, scratch, scratch + total);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// backward operand: B_z[f, o] = weight[(f*K + z)*Fo + o]  (f < F rows of G_z, o < Fo contraction)
int fused_bwd_prep(const float* weight, int F, int Fo, int K, float* scratch, cudaStream_t st) {
  const int N = ft::pad16(F), Kp = ft::pad32(Fo);
  const long long total = (long long)K * N * Kp;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 1184);
  ft::prep_w_kernel<<<blocks, 256, 0, st>>>(weight, (long long)K * Fo, 1, Fo, F, Fo, N, Kp, K, scratch, scratch + total);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace agcn
