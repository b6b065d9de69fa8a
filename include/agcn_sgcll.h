/*
 * agcn_sgcll.h -- C ABI of libagcn_sm100.so: the SGC-LL hot path of
 * uta-smile/Adaptive-Graph-Convolutional-Network on NVIDIA B200 (sm_100a).
 *
 * The reference has no FFI layer (it is 100 % Python on TensorFlow 0.12); the
 * boundary below is what a maintainer would bind from the Python layer classes
 * (ctypes stub in INTEGRATION.md).  Each entry point cites the reference code it
 * replaces, paths relative to the reference root.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; nothing is
 *     allocated inside the compute calls; all work is ordered on `stream`
 *     (a cudaStream_t passed as void*).
 *   - return value: 0 = AGCN_OK, negative = AGCN_ERR_*; agcn_last_error() gives
 *     the text for the calling thread.
 *   - all floating point data is IEEE fp32, indices int32, Laplacian offsets int64.
 *   - thread-safe for distinct plans / streams.
 *
 * Native HBM layout ("packed"): a batch of B graphs with n_g real nodes is stored
 * without padding.  Node matrices are [R, F] row-major with R = sum n_g, graph g
 * owning rows node_off[g] .. node_off[g+1]-1; per-graph n_g x n_g matrices
 * (Laplacians) are stored back to back, graph g at element offset
 * lap_off[g] = sum_{h<g} n_h^2 with leading dimension n_g.  The reference's wire
 * layout (zero-padded [B, Nmax, F] / [B, Nmax, Nmax],
 * models/tf_modules/graph_topology.py:84-98) is converted at the boundary by
 * agcn_pack_* / agcn_unpack_*; padded rows come back as exact +0.0f.
 */
#ifndef AGCN_SGCLL_H_
#define AGCN_SGCLL_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGCN_OK 0
#define AGCN_ERR_INVALID (-1)   /* bad argument / unsupported shape            */
#define AGCN_ERR_CUDA (-2)      /* a CUDA runtime call failed                  */
#define AGCN_ERR_WORKSPACE (-3) /* workspace too small                         */
#define AGCN_ERR_NO_DEVICE (-4) /* no sm_100 device / kernel image unusable    */

/* layer variant: models/layers/graphconv.py:32 / graphconv_reslap.py:15 */
#define AGCN_VARIANT_SGC_LL 0
#define AGCN_VARIANT_SGC_LL_RESLAP 1
/* SURVEY.md section 0 (Q2): what `L = I - D * W * D` means */
#define AGCN_LAP_REFERENCE_LITERAL 0 /* elementwise on ndarrays => res_L == I (graphconv.py:198-200) */
#define AGCN_LAP_PAPER 1             /* I - D^-1/2 W D^-1/2                                          */
/* SURVEY.md section 0 (Q1): tf.py_func has no gradient (graphconv.py:211) */
#define AGCN_METRIC_GRAD_REFERENCE 0 /* stop-gradient through the metric block */
#define AGCN_METRIC_GRAD_FULL 1      /* differentiable metric (paper)          */
/* activation fused into the output epilogue (graphconv.py:118-123); others are applied by the host */
#define AGCN_ACT_LINEAR 0
#define AGCN_ACT_RELU 1

/* optional outputs (graphconv.py:125 returns res_L and res_W lists; graphconv_reslap.py:89 adds L_all) */
#define AGCN_OUT_RES_L 1u
#define AGCN_OUT_RES_W 2u
#define AGCN_OUT_L_ALL 4u
#define AGCN_SAVE_FOR_BACKWARD 8u /* forward keeps what backward needs in `d_saved` */

typedef struct agcn_plan agcn_plan; /* opaque: topology of one batch */

typedef struct agcn_sgcll_desc {
  int32_t F;              /* input features  (n_atom_feature, graphconv.py:58)  */
  int32_t Fo;             /* output features (nb_filter,      graphconv.py:57)  */
  int32_t K;              /* Chebyshev order (graphconv.py:61), >= 1            */
  int32_t variant;        /* AGCN_VARIANT_*                                     */
  int32_t laplacian_mode; /* AGCN_LAP_*                                         */
  int32_t metric_grad;    /* AGCN_METRIC_GRAD_*                                 */
  int32_t activation;     /* AGCN_ACT_*                                         */
  uint32_t flags;         /* AGCN_OUT_* | AGCN_SAVE_FOR_BACKWARD                */
} agcn_sgcll_desc;

/* ---- library ---------------------------------------------------------- */
int agcn_version(void);
const char* agcn_last_error(void);
/* number of kernels this library has launched so far in this process (bench.py's gpu_launches) */
uint64_t agcn_launch_count(void);

/* ---- batch topology (replaces GraphTopologyMol.batch_to_feed_dict's data_slice / lap_slice,
 *      models/tf_modules/graph_topology.py:100-135) ----------------------------------------- */
/* n_nodes_host[B]: real node count of every graph (host memory, 1 <= n_g <= Nmax).
 * Builds the device-side offset tables and the work lists (size-sorted graphs, 128-row tiles).  The tables are
 * uploaded in stream order on `stream` (stream-ordered allocation, pooled pinned staging, pooled side streams):
 * nothing is synchronised, so a plan per training batch costs tens of microseconds of host time.  Calls that use
 * the plan on another stream are ordered after the upload automatically.  agcn_plan_destroy may be called as
 * soon as the last call using the plan has returned; the device block is released in stream order. */
int agcn_plan_create(const int32_t* n_nodes_host, int32_t B, int32_t Nmax, void* stream, agcn_plan** out);
int agcn_plan_destroy(agcn_plan* plan);
int64_t agcn_plan_total_nodes(const agcn_plan* plan);    /* R = sum n_g      */
int64_t agcn_plan_total_lap(const agcn_plan* plan);      /* sum n_g^2        */
const int32_t* agcn_plan_node_off_host(const agcn_plan* plan); /* [B+1] host   */
const int64_t* agcn_plan_lap_off_host(const agcn_plan* plan);  /* [B+1] host   */

/* Host-only view of the work decomposition of the fused tile kernels (no reference counterpart; exported for
 * tests and tuning): the graphs of a batch are packed into 128-row tiles.  Tile t owns entries
 * gstart[t] .. gstart[t+1]; an entry is 4 int32: {graph, first tile row, n_g, offset of the graph's matrix in
 * the tile's shared-memory Laplacian area} for a whole graph, or {graph, first graph row, rows, -1} for a
 * 128-row range of a graph too large to share a tile.  Call with NULL buffers to get the counts. */
int agcn_fused_tiles_host(const int32_t* n_nodes_host, int32_t B, int32_t* gstart_out, int32_t gstart_cap,
                          int32_t* entries_out, int32_t entries_cap, int32_t* tiles_out, int32_t* n_entries_out);

/* Measurement aid (no reference counterpart; bench.py's roofline): while enabled, every eager agcn_sgcll_forward on
 * the tile path brackets the launch of its tensor-core contraction with CUDA events on the launching stream;
 * agcn_fused_profile_read waits for them and returns the summed duration (ms) and the number of launches since
 * the last read.  Must be off during CUDA graph capture. */
int agcn_fused_profile(int enable);
int agcn_fused_profile_read(float* ms_sum, int* launches);

/* The same for every main kernel of the library (bench.py's per-kernel roofline table): while enabled (and the stream
 * is not capturing) the host wrappers bracket each launch with CUDA events on its stream.  agcn_profile_read waits
 * for them, clears the records and writes one line per kernel, "name<TAB>launches<TAB>milliseconds\n", into buf
 * (NUL-terminated, truncated to cap); *needed receives the size the whole table takes. */
int agcn_profile_enable(int enable);
int agcn_profile_read(char* buf, size_t cap, size_t* needed);
/* The same records as a timeline instead of sums: one line per launch, "name<TAB>start_ms<TAB>end_ms\n", times relative
 * to the start of the first recorded launch (the streams of a step overlap: this shows what is on the critical path). */
int agcn_profile_timeline(char* buf, size_t cap, size_t* needed);
/* fp32-FMA peak probe for the roofline denominators (SURVEY.md section 8d asks for a measured fp32 peak next to the
 * recorded bf16 one): 148 x 8 CTAs of 256 threads, 8 independent FMA chains of `iters` trips per thread, i.e.
 * 148 * 8 * 256 * 8 * 2 * iters FLOP; d_sink needs 148 * 8 * 256 floats.  The caller times it with CUDA events. */
int agcn_probe_fp32_fma(float* d_sink, int32_t iters, void* stream);

/* Tuning aid (no reference counterpart): d_buf = device buffer of tiles x 128 uint64; the following fused forward
 * launches record a per-tile timeline of nanosecond stamps into it.  NULL switches the recording off. */
int agcn_fused_debug_set(void* d_buf);

/* Tuning / debugging aid (no reference counterpart): Out = cmul * op(L_g) In over the rows of every graph with more
 * than AGCN_CHEB_SMALL_MAX nodes (the row-tiled path; other rows of Out are not written), op = L (+I) or L^T (+I);
 * impl 0 = the library's own choice, 1 = SIMT kernel, 2 = tcgen05 kernel (F % 4 == 0, F >= 16), 3 = streaming kernel
 * (F <= 8), 4 = the equal-size-graph tcgen05 kernel (n % 128 == 0 for every graph of the batch) whatever the grid size.
 * tools/dbg_grouped.py compares the implementations block by block. */
int agcn_debug_grouped_product(const agcn_plan* plan, const float* d_L /*packed*/, const float* d_In /*[R,F]*/,
                               float* d_Out /*[R,F]*/, int32_t F, int32_t transL, int32_t add_identity, float cmul,
                               int32_t impl, void* stream);

/* d_buf = device buffer of 1024 uint64 (or NULL): the following agcn_debug_grouped_product calls with impl 2 record a
 * nanosecond timeline of their first CTA into it (tools/tc_timeline.py). */
int agcn_debug_grouped_timeline(void* d_buf);

/* ---- layout conversion (pad_data2sparse / pad_Lap2sparse, graph_topology.py:84-98;
 *      tf.slice at graphconv.py:153-154; tf.pad at graphconv.py:249-251) ------------------ */
int agcn_pack_nodes(const agcn_plan* plan, const float* d_padded /*[B,Nmax,F]*/, float* d_packed /*[R,F]*/,
                    int32_t F, void* stream);
int agcn_unpack_nodes(const agcn_plan* plan, const float* d_packed, float* d_padded, int32_t F, void* stream);
int agcn_pack_lap(const agcn_plan* plan, const float* d_padded /*[B,Nmax,Nmax]*/, float* d_packed, void* stream);
int agcn_unpack_lap(const agcn_plan* plan, const float* d_packed, float* d_padded, void* stream);
/* The same packed matrices from the CSR form Graph.compute_laplacian produces (graph_structure.py:100-107), so the
 * dense [Nmax,Nmax] padding of pad_Lap2sparse never exists: d_indptr [R+1] row pointers over the packed rows of the
 * whole batch, d_indices column inside the row's own graph, d_values fp32 (SURVEY.md section 8f row 2). */
int agcn_pack_lap_csr(const agcn_plan* plan, const int32_t* d_indptr, const int32_t* d_indices, const float* d_values,
                      float* d_packed, void* stream);

/* ---- graph construction for point clouds on the device (SURVEY.md section 8f row 4): the threshold adjacency of the
 * reference's loaders, then Graph.compute_laplacian (models/graph_structure.py:85-130), for a whole packed batch.
 *   AGCN_ADJ_MEAN_DISTANCE  utils/data_loader/meshloader.py:264-285: i ~ j iff d_ij < mean distance over the pairs j <= i
 *   AGCN_ADJ_CUTOFF         utils/data_loader/pointcloudloader.py:240-263: d_lim = the int(n * sparse_ratio)-th largest
 *                           distance (np.sort(all_dist)[-cut_off_idx]; index -0 = the smallest = 0: no edges)
 * d_points [R, F] packed coordinates (1 <= F <= 8; the distance uses all F columns, like the reference), d_L packed
 * float32 Laplacians out (what batch_to_feed_dict would feed as 'original_laplacian').  The n x n distance matrix is
 * never stored: every sweep recomputes it from the coordinates. */
#define AGCN_ADJ_MEAN_DISTANCE 0
#define AGCN_ADJ_CUTOFF 1
int agcn_point_laplacian_workspace_bytes(const agcn_plan* plan, size_t* bytes);
int agcn_point_laplacian(const agcn_plan* plan, const float* d_points, int32_t F, int32_t rule, float sparse_ratio,
                         float* d_L, void* d_work, size_t work_bytes, void* stream);

/* ---- GraphPoolMol (graphpool.py:55-110; SURVEY.md section 8f row 4) ------------------------
 * Y[i,:] = max over {j : L[i,j] != 0} of X[j,:] per graph (a row without a non-zero keeps X[i,:]).  d_argmax
 * (optional, [R,F] int32) receives the packed row that supplied each maximum.  The reference computes this inside
 * tf.py_func (no gradient); agcn_graph_pool_backward is the arg-max gradient for callers that want one:
 * dX[argmax[r,f], f] += dY[r,f]. */
int agcn_graph_pool(const agcn_plan* plan, const float* d_X /*[R,F]*/, const float* d_L /*packed*/, float* d_Y,
                    int32_t* d_argmax, int32_t F, void* stream);
int agcn_graph_pool_backward(const agcn_plan* plan, const float* d_dY, const int32_t* d_argmax, float* d_dX, int32_t F,
                             void* stream);

/* ---- SGC-LL layer ----------------------------------------------------- */
/* sizes in BYTES of the two scratch areas: `saved` lives from forward to backward, `work` only
 * inside one call (max of forward and backward). */
int agcn_sgcll_workspace_bytes(const agcn_sgcll_desc* desc, const agcn_plan* plan, size_t* saved_bytes,
                               size_t* work_bytes);

/* SGC_LL.specgraph_LL (graphconv.py:127-252) / SGC_LL_Reslap.specgraph_LL_reslap
 * (graphconv_reslap.py:91-230) plus the activation of call() (graphconv.py:118-123), whole batch.
 *   d_X      [R,F]        node features (packed)
 *   d_Lint   [sum n^2]    intrinsic Laplacians (packed)            'original_laplacian'
 *   d_Lprev  [sum n^2]    Reslap: previous layer's L_all or NULL   'res_lap'
 *   d_M_L [F,F], d_weight [F*K,Fo] (row f*K+k), d_bias [Fo], d_alpha [1], d_beta [1] (Reslap, else NULL)
 *   d_Y      [R,Fo]       activated output (packed)
 *   d_resL / d_resW / d_Lall [sum n^2]  optional outputs (NULL unless the flag is set; d_Lall is
 *                                       mandatory for Reslap when AGCN_OUT_L_ALL is set)
 */
int agcn_sgcll_forward(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                       const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_bias,
                       const float* d_alpha, const float* d_beta, float* d_Y, float* d_resL, float* d_resW,
                       float* d_Lall, void* d_saved, void* d_work, size_t work_bytes, void* stream);

/* Gradient of the above (what tf.gradients builds for graphconv.py:212-251; PyFunc => no gradient
 * through the metric unless metric_grad == FULL).
 *   d_dY       [R,Fo]      gradient w.r.t. the activated output
 *   d_dLall_in [sum n^2]   Reslap: gradient flowing into the returned L_all from later layers, or NULL
 *   outputs: d_dX [R,F], d_dM_L [F,F], d_dweight [F*K,Fo], d_dbias [Fo], d_dalpha [1], d_dbeta [1] (Reslap),
 *            d_dLprev [sum n^2] (Reslap with d_Lprev, else NULL).  All outputs are overwritten.
 *            d_dX may be NULL when the caller does not need it (first layer: the atom features have no gradient).
 */
int agcn_sgcll_backward(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                        const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_alpha,
                        const float* d_beta, const float* d_Y, const float* d_dY, const float* d_dLall_in,
                        const void* d_saved, float* d_dX, float* d_dM_L, float* d_dweight, float* d_dbias,
                        float* d_dalpha, float* d_dbeta, float* d_dLprev, void* d_work, size_t work_bytes,
                        void* stream);

/* Building block of the backward pass, exported for unit tests and tuning (no reference counterpart: it is
 * the dW = T^T dY contraction that tf.gradients derives from graphconv.py:245-247):
 *   out[(f*S + s)*N + c] = sum_r A_s[r, f] * D[r, c],  A_0 = d_A0 [M,Kd], A_s = d_A1 + (s-1)*M*Kd, D [M,N].
 * use_tensor_cores: 1 = tcgen05 3xTF32 kernel (needs Kd <= 128, Kd % 4 == 0, N % 4 == 0), 0 = CUDA cores. */
size_t agcn_gemm_tn_scratch_bytes(int32_t M, int32_t Kd, int32_t N, int32_t S);
int agcn_gemm_tn(const float* d_A0, const float* d_A1, const float* d_D, float* d_out, int32_t M, int32_t Kd,
                 int32_t N, int32_t S, void* d_scratch, int32_t use_tensor_cores, void* stream);

/* Node-level linear map over the packed rows:  C (+)= act(scale * A op(B) + bias),  A [M,Kd] (row pitch lda),
 * op(B) = B [Kd,N] or, transB, B^T with B [N,Kd]; d_scale = optional DEVICE scalar (a learned beta), d_bias [N] optional.
 * The per-graph matmuls of BlockEnd (models/layers/blockend.py:67-86), DenseBlockEnd (densenet_block.py:98-131), MLP
 * (MLP.py:69-83) and DenseMol (dense_layer.py:33-50) are this product over all R rows at once; tcgen05 3xTF32 when the
 * operands are TMA-compatible (Kd >= 32, 16-byte pitches), CUDA cores otherwise.  Scratch:
 * agcn_node_gemm_scratch_bytes(N, Kd) bytes. */
size_t agcn_node_gemm_scratch_bytes(int32_t N, int32_t Kd);
int agcn_node_gemm(const float* d_A, int32_t lda, const float* d_B, int32_t ldb, int32_t transB, float* d_C, int32_t ldc,
                   int32_t M, int32_t N, int32_t Kd, const float* d_bias, const float* d_scale, int32_t accumulate,
                   int32_t activation, void* d_scratch, void* stream);

/* Dropout of the layer output in the train phase (models/layers/dropout.py:27-41 -> tf.nn.dropout(x, 1 - p, seed);
 * graphconv.py:121-122): y[i] = keep_i ? x[i] / (1 - p) : 0 with keep_i from a counter-based Philox4x32-10 stream
 * keyed by (seed, i).  Nothing is stored: the same call on dY with the same seed is the gradient.  d_Y may alias d_X. */
int agcn_dropout(const float* d_X, float* d_Y, int64_t n, float p, uint64_t seed, void* stream);

/* Labels as the reference feeds them (multitask_classifier.py:147-152,171-185: y[b, t] in {0, 1}, w[b, t]) -> the
 * [B, 2 n_tasks] one-hot targets (tf.one_hot(label, 2), multitask_classifier.py:196-199) and per-logit weights that
 * agcn_head_loss_grad reads.  y / w may be device pointers or PINNED host pointers (read in place over PCIe). */
int agcn_expand_labels(const uint8_t* y, const float* w, int32_t B, int32_t n_tasks, float* d_targets, float* d_weights,
                       void* stream);

/* ---- the layers after the last SGC-LL layer (SURVEY.md section 8f, rows 1 and 3), loss and gradient in one call:
 *   DenseMol (models/layers/dense_layer.py:33-50, linear) + GraphGatherMol (models/layers/graphgather.py:50-78:
 *   per-graph sum over the real atoms, tanh) + the n_tasks two-class heads (models/operators/model_operatos.py:
 *   792-864) as one [Fm, Nt = 2 n_tasks] matrix + weighted sigmoid cross-entropy summed and multiplied by `scale`
 *   (= 1 / global batch size, models/tf_modules/multitask_classifier.py:41-44,187-209).
 *   d_H [R,Fh] packed output of the last SGC-LL layer; d_dense_W [Fh,Fm], d_dense_b [Fm]; d_head_W [Fm,Nt],
 *   d_head_b [Nt]; d_targets / d_weights [B,Nt].
 *   outputs (overwritten): d_loss [1], d_dH [R,Fh] and the four parameter gradients.
 *   Needs Fm >= 32 and a multiple of 4 (the logits contraction runs on the tensor cores with the loss as its
 *   epilogue); the other contractions fall back to CUDA-core kernels when their shape is not TMA-compatible.
 *
 *   agcn_head_loss_grad_ex adds `loss_kind`: AGCN_LOSS_SIGMOID_CE (the multitask head above),
 *   AGCN_LOSS_SOFTMAX_CE = the single-task multi-class head of SingletaskGraphClassifier
 *   (models/tf_modules/singletask_classifier.py:124-151, get_loss_fn('softmax_cross_entropy') of
 *   multitask_classifier.py:45-48): Nt = n_classes, d_targets [B,Nt] one-hot, d_weights [B] per-sample weights,
 *   loss = scale * sum_b w_b (logsumexp(x_b) - <y_b, x_b>), or
 *   AGCN_LOSS_WEIGHTED_L2 = the regression head of MultitaskGraphRegressor (models/tf_modules/multitask_regressor.py,
 *   DeepChem 1.x, default final_loss='weighted_L2'; restated, parity unpinned): Nt = n_tasks, head_W [Fm,Nt] is one
 *   [Fm,1] fully connected layer per task side by side, x[b,t] = (mol head_W + head_b)[b,t] with no activation,
 *   d_targets / d_weights [B,Nt] float (no label expansion),
 *   loss = scale * sum_b sum_t (w[b,t] (x[b,t] - y[b,t]))^2, d loss / d x = 2 w^2 (x - y) scale.  The weight enters
 *   squared (tf.square(tf.mul(tf.sub(x, t), w))): with 0/1 weights masking missing labels that is w (x - y)^2.  The loss
 *   and its gradient are the epilogue of the output GEMM, as for the sigmoid heads. */
#define AGCN_LOSS_SIGMOID_CE 0
#define AGCN_LOSS_SOFTMAX_CE 1
#define AGCN_LOSS_WEIGHTED_L2 2
int agcn_head_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t Fm, int32_t Nt, size_t* bytes);
int agcn_head_loss_grad(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                        const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                        float scale, int32_t Fh, int32_t Fm, int32_t Nt, float* d_loss, float* d_dH,
                        float* d_ddense_W, float* d_ddense_b, float* d_dhead_W, float* d_dhead_b, void* d_work,
                        size_t work_bytes, void* stream);

int agcn_head_loss_grad_ex(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                           const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                           float scale, int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_loss,
                           float* d_dH, float* d_ddense_W, float* d_ddense_b, float* d_dhead_W, float* d_dhead_b,
                           void* d_work, size_t work_bytes, void* stream);

/* Prediction with the same head (the forward half of agcn_head_loss_grad_ex, no gradient): what predict_proba of
 * MultitaskGraphClassifier / SingletaskGraphClassifier returns (models/tf_modules/multitask_classifier.py,
 * singletask_classifier.py; parity unpinned, as the other TensorFlow ops of DESIGN.md section 7).
 *   AGCN_LOSS_SIGMOID_CE: Nt = 2 n_tasks, column 2t+c = class c of task t; probs[b, 2t+c] is the softmax over that task's
 *     two logits, 1 / (1 + exp(x[2t+1-c] - x[2t+c])) -- read as [B, n_tasks, 2], the layout of DeepChem's
 *     MultitaskGraphClassifier.predict_proba (a softmax over every task's [B, 2] logits).  Nt must be even.  The
 *     probabilities are the epilogue of the logits GEMM: the logits never reach memory.
 *   AGCN_LOSS_SOFTMAX_CE: probs[b, :] = softmax over the Nt class logits.
 *   AGCN_LOSS_WEIGHTED_L2: d_probs receives the regression values x [B, Nt = n_tasks] themselves (predict of
 *     MultitaskGraphRegressor), written by the output GEMM's epilogue; there is no probability.
 *   d_probs [B,Nt] out.  d_targets / d_weights / d_loss are all NULL, or all set: then d_loss [1] also receives the
 *   weighted loss x scale, bit-identical to the loss agcn_head_loss_grad_ex writes for the same inputs.
 *   Same size rules as agcn_head_loss_grad_ex (Fm >= 32 and a multiple of 4). */
int agcn_head_predict_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t Fm, int32_t Nt, size_t* bytes);
int agcn_head_predict(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                      const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                      float scale, int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_probs, float* d_loss,
                      void* d_work, size_t work_bytes, void* stream);

/* ---- one training step's loss and gradients as ONE call: the counterpart of `sess.run([train_op, loss, ...])`
 *      (models/tf_modules/multitask_classifier.py:255-264), which executes the whole graph of
 *      models/networks/basic_AGCN.py:35-47 inside the TensorFlow runtime.  A stack = n_layers SGC_LL layers (relu or
 *      linear activation, any semantics modes) + DenseMol + GraphGatherMol + logits + loss; the call chains
 *      agcn_sgcll_forward / agcn_head_loss_grad_ex / agcn_sgcll_backward over one arena.
 *   param_offsets: element offsets into the flat parameter buffer (and, identically, the flat gradient buffer):
 *      5 per layer {weight [F*K,Fo], bias [Fo], M_L [F,F], alpha [1], -1}, then dense_W [Fh,Fm], dense_b [Fm],
 *      head_W [Fm,Nt], head_b [Nt].
 *   notify (optional): called on the host right after the gradients of a stage have been ENQUEUED on `stream`
 *      (stage n_layers = head + dense, then n_layers-1 .. 0 = that SGC_LL layer), so a data-parallel caller can start
 *      the all-reduce of a gradient bucket while the earlier layers are still running backward. */
typedef struct agcn_stack agcn_stack;
typedef void (*agcn_stack_notify_fn)(void* user, int32_t stage, void* stream);
int agcn_stack_create(const agcn_sgcll_desc* layer_descs, int32_t n_layers, int32_t Fm, int32_t Nt, int32_t loss_kind,
                      const int64_t* param_offsets, agcn_stack** out);
int agcn_stack_destroy(agcn_stack* stack);
int agcn_stack_workspace_bytes(const agcn_stack* stack, const agcn_plan* plan, size_t* bytes);
int agcn_stack_loss_grad(const agcn_stack* stack, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                         const float* d_targets, const float* d_weights, float scale, const float* d_params,
                         float* d_grads, float* d_loss, void* d_work, size_t work_bytes, agcn_stack_notify_fn notify,
                         void* notify_user, void* stream);
/* Forward-only counterpart of agcn_stack_loss_grad (predict_proba / evaluate of the reference's classifiers, predict /
 * evaluate of its regressor): the layers run without AGCN_SAVE_FOR_BACKWARD, then agcn_head_predict.  d_probs [B,Nt] as
 * agcn_head_predict (the values x for AGCN_LOSS_WEIGHTED_L2); d_targets /
 * d_weights / d_loss all NULL or all set (then d_loss [1] is bit-identical to agcn_stack_loss_grad's loss for the same
 * batch, parameters and scale).  Nothing outside d_probs, d_loss and d_work is written; no allocation, no
 * synchronisation, no host callback (capturable).  The arena holds two [R, max Fo] activation buffers and ONE `saved`
 * area that each layer reuses, so it is smaller than agcn_stack_workspace_bytes'. */
int agcn_stack_predict_workspace_bytes(const agcn_stack* stack, const agcn_plan* plan, size_t* bytes);
int agcn_stack_predict(const agcn_stack* stack, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                       const float* d_targets, const float* d_weights, float scale, const float* d_params,
                       float* d_probs, float* d_loss, void* d_work, size_t work_bytes, void* stream);

/* ---- residual networks in the same calls: a stack described as a list of nodes.  Node i takes H[i-1] as input (node 0
 *      takes d_X); the last node's output feeds the head.  This is ResidualGraphMolResLap of the reference
 *      (models/networks/tf_graphs.py:159-223): SGC_LL_Reslap layers whose L_prev is an earlier Reslap layer's L_all
 *      (L_all = leaky_a(clip(leaky_a(clip(res_L)) + L_int + beta L_prev)), graphconv_reslap.py:91-230) and BlockEnd
 *      nodes that close a residual block (blockend.py:67-86).
 *   AGCN_NODE_SGCLL      an SGC_LL layer (desc.variant AGCN_VARIANT_SGC_LL, src -1) or an SGC_LL_Reslap layer
 *                        (AGCN_VARIANT_SGC_LL_RESLAP; src = the earlier Reslap node whose L_all is its L_prev, or -1 for
 *                        res_lap = []).  desc.flags is ignored: the stack sets what the layer classes set.
 *   AGCN_NODE_BLOCK_END  H[i] = act(H[src] W + H[i-1]), act = desc.activation (relu or linear); desc.F = width of
 *                        H[src], desc.Fo = width of H[i-1], the other desc fields 0.
 *   param_offsets: 5 per node, then the 4 head tensors, as agcn_stack_create: SGC_LL {weight, bias, M_L, alpha, -1},
 *      Reslap {weight, bias, M_L, alpha, beta}, BlockEnd {weight [F, Fo], -1, -1, -1, -1}.
 *   Rejected (AGCN_ERR_INVALID, agcn_last_error names the node): an unknown kind or variant, a BlockEnd as node 0, a
 *      src that is not an earlier node, a Reslap src that is not a Reslap node, two Reslap nodes or two BlockEnds
 *      naming the same src, widths that do not chain, a Reslap node without a beta offset, an SGC_LL node with a src.
 *   agcn_stack_workspace_bytes, agcn_stack_loss_grad, agcn_stack_predict(_workspace_bytes) and agcn_stack_destroy take
 *   either kind of stack.  notify stages: n_nodes = head + dense, then node i's parameters, last node first.  The calls
 *   chain agcn_sgcll_forward / agcn_sgcll_backward, agcn_node_gemm, agcn_gemm_tn and the head calls with the arguments
 *   the layer classes pass them, so their results equal the layer classes' under torch.autograd bit for bit.  The
 *   training arena keeps every node's output and `saved` area, one L_all per Reslap node and the gradients the
 *   dependencies need; the prediction arena reuses activation and L_all slots once their last reader has run.
 *   agcn_stack_create(descs, n, ...) is agcn_stack_create_nodes with every node an SGC_LL layer and src = -1. */
#define AGCN_NODE_SGCLL 0
#define AGCN_NODE_BLOCK_END 1
typedef struct agcn_stack_node {
  int32_t kind;           /* AGCN_NODE_*                                                                   */
  agcn_sgcll_desc desc;   /* the layer (SGCLL) or {F, Fo, 0, 0, 0, 0, activation, 0} (BLOCK_END)          */
  int32_t src;            /* Reslap: the L_prev producer or -1; BLOCK_END: the node whose output is x_res  */
} agcn_stack_node;
int agcn_stack_create_nodes(const agcn_stack_node* nodes, int32_t n_nodes, int32_t Fm, int32_t Nt, int32_t loss_kind,
                            const int64_t* param_offsets, agcn_stack** out);

/* tf.train.AdamOptimizer's update (multitask_classifier.py:233-237) over a flat parameter buffer:
 *   t = *d_step + 1;  lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t);  m = beta1 m + (1 - beta1) g;
 *   v = beta2 v + (1 - beta2) g^2;  p -= lr_t m / (sqrt(v) + eps);  *d_step = t.
 * The step counter lives on the device so that a captured CUDA graph of the step replays correctly. */
int agcn_adam_step(float* d_params, const float* d_grads, float* d_m, float* d_v, int32_t* d_step, int64_t n, float lr,
                   float beta1, float beta2, float eps, void* stream);

/* One graph launch per training step for batches whose topology changes every step.
 * Eager launches of the ~80 kernels of a step are what bulk host->device traffic hurts: the next batch arriving over
 * PCIe delays the front end's fetch of every launch command (0.70 -> 0.82 ms per ToxCast step), while a graph launch of
 * the same step is not affected at all (tools/replay_vs_pcie.py).  A captured graph cannot simply be replayed for a new
 * batch (grid sizes, tile tables and buffers differ), so the step is RE-CAPTURED for every batch -- capture submits no
 * work, it costs the host what the launches cost -- and an executable graph kept from the previous step is updated in
 * place with the new kernel parameters (cudaGraphExecUpdate: same nodes, new arguments and grids) and launched once.
 * When the node topology itself differs (another set of size buckets) the executable graph is instantiated anew.
 *   agcn_capture_begin(stream);  ... the library calls of the step on `stream` ...;  agcn_capture_end_launch(stream, &g, &how);
 * *how: 1 = updated in place, 0 = instantiated (first use), -r = instantiated after the update of the most recent
 * executable graph was refused with cudaGraphExecUpdateResult r (2 = topology changed, 4 = function changed, ...).  The plan of the batch must have been created (and its upload ordered
 * before `stream`) outside the capture. */
typedef struct agcn_step_graph agcn_step_graph;
int agcn_capture_begin(void* stream);
int agcn_capture_end_launch(void* stream, agcn_step_graph** graph /* in/out, *graph == NULL the first time */,
                            int32_t* how);
int agcn_capture_abort(void* stream);   /* after a failed call inside the capture: end it and drop what was recorded */
int agcn_step_graph_destroy(agcn_step_graph* graph);

/* Host-buffer convenience entry (the end-to-end path): padded HOST arrays in the reference's wire
 * layout in, padded HOST output out; host<->device copies are issued on `stream` inside the call.
 * Page-locked inputs (cudaMallocHost / cudaHostRegister / torch pin_memory) are read in place by the pack kernels
 * (only the real rows cross PCIe); pageable inputs are staged through the copy engine.
 * d_scratch must hold agcn_sgcll_host_scratch_bytes() bytes of device memory. */
int agcn_sgcll_host_scratch_bytes(const agcn_sgcll_desc* desc, const agcn_plan* plan, size_t* bytes);
int agcn_sgcll_forward_host(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* h_X_padded,
                            const float* h_L_padded, const float* d_M_L, const float* d_weight, const float* d_bias,
                            const float* d_alpha, float* h_Y_padded, void* d_scratch, size_t scratch_bytes,
                            void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGCN_SGCLL_H_ */
