/*
 * flowcompare_b200 -- C ABI of the B200-native per-point conditional log-likelihood path.
 *
 * This is the drop-in boundary for the hot path of SamGalanakis/FlowCompare
 * (reference `model_initialization.py:206-228` `inner_loop` and everything below it).
 * The reference's own native boundary is a set of `extern "C"` launchers taking raw device
 * pointers, explicit int dims and a `cudaStream_t`
 * (e.g. `models/scene_seg_PAConv/lib/pointops/src/knnquery_heap/knnquery_heap_cuda_kernel.h:10-18`),
 * wrapped by pybind (`lib/pointops/src/pointops_api.cpp:15-40`).  The entry points below keep that
 * convention -- caller allocates every output, plain pointers + sizes, no torch types -- but
 *   - return an int status (0 = FC_OK, negative = error) instead of `exit(-1)`
 *     (reference `lib/pointops/src/grouping/grouping_cuda_kernel.cu:87-91`);
 *   - never allocate: scratch memory is passed in (`*_workspace_bytes` queries);
 *   - launch everything on the stream passed in (several reference kernels use the legacy
 *     default stream, e.g. `lib/pointops/src/sampling/sampling_cuda_kernel.cu:40`).
 *
 * All pointers are DEVICE pointers unless the name ends in `_host`.  All matrices are row-major
 * fp32; point clouds are [B, N, C] (point-major), the layout `inner_loop` receives.
 * There is no CPU fallback anywhere in this library.
 */
#ifndef FLOWCOMPARE_B200_H
#define FLOWCOMPARE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* fc_stream_t; /* a cudaStream_t */

#if defined(__GNUC__)
#define FC_API __attribute__((visibility("default")))
#else
#define FC_API
#endif

enum {
    FC_OK = 0,
    FC_ERR_INVALID_ARG = -1,
    FC_ERR_CUDA = -2,       /* a CUDA runtime call failed; see fc_last_error() */
    FC_ERR_LAUNCH = -3,     /* a kernel launch failed; see fc_last_error() */
    FC_ERR_WORKSPACE = -4,  /* workspace too small / misaligned */
    FC_ERR_UNSUPPORTED = -5,
    FC_ERR_MODEL = -6       /* model description inconsistent */
};

FC_API int fc_version(void);
/* Human-readable description of the last error raised on this thread ("" if none). */
FC_API const char* fc_last_error(void);

/* ------------------------------------------------------------------ kNN ------------------
 * fc_knn_self replaces `knn(x, k)` of reference models/pytorch_gcn.py:13-20 (called from
 * get_graph_feature :27): for every point the k nearest points of the SAME cloud (self included)
 * in ascending squared distance.  x is [B, N, ldx] with the C feature columns used starting at
 * column 0.  Arithmetic (the "canonical form" the bit-exact oracle oracle/knn_ref.c restates):
 *   dot_ij = fmaf chain over c = 0..C-1;  xx_i likewise;  pd_ij = ((-xx_j) - (-2*dot_ij)) - xx_i
 * (the reference's algebraic form, fixed summation order); the k LARGEST pd are selected, ties
 * broken by LOWER index.  idx32 [B,N,k] and idx64 [B,N,k] are both optional (NULL to skip one).
 * Requires 1 <= k <= 64 and k <= N.                                                           */
FC_API int fc_knn_self(const float* x, int ldx, int B, int N, int C, int k,
                int32_t* idx32, int64_t* idx64, fc_stream_t stream);

/* fc_knn_query replaces `get_knn(samples, context_cloud, n_neighbors)` / `KNN_torch_fun` of
 * reference knn.py:40-52,79-90: queries q [Nq, D], train t [Nt, D] -> idx64 [Nq, k], ascending
 * diss_ij = (qq_i + tt_j) - 2*dot_ij, ties by lower index.  1 <= k <= 64, k <= Nt.
 * With k = 1 and t = the voxel-centre grid it is also the label pass of `voxelize(pos, start, end, size)`
 * (reference utils.py:446-454, called by dataloaders/ams_voxel_loader.py:204).                 */
FC_API int fc_knn_query(const float* q, const float* t, int Nq, int Nt, int D, int k,
                 int64_t* idx64, fc_stream_t stream);

/* Workspace forms of the two entry points above.  fc_knn_self / fc_knn_query keep the round-1 signatures (no workspace
 * argument) and are the ONE exception to "never allocate": they use a per-device scratch (norms + distance keys) that
 * grows on demand, so two calls on different streams of the same device must not overlap.  The _ws forms take the
 * scratch from the caller (fc_knn_workspace_bytes(B, Nq, Nt, self): B clouds, self = 1 for fc_knn_self_ws with
 * Nq = Nt = N, self = 0 and B = 1 for fc_knn_query_ws), touch no global state and are independent per stream.
 * FC_ERR_WORKSPACE if the workspace is NULL or too small.  Results are identical to the forms above.            */
FC_API int64_t fc_knn_workspace_bytes(int B, int Nq, int Nt, int self);
FC_API int fc_knn_self_ws(const float* x, int ldx, int B, int N, int C, int k, int32_t* idx32, int64_t* idx64,
                   void* workspace, int64_t workspace_bytes, fc_stream_t stream);
FC_API int fc_knn_query_ws(const float* q, const float* t, int Nq, int Nt, int D, int k, int64_t* idx64,
                    void* workspace, int64_t workspace_bytes, fc_stream_t stream);

/* ------------------------------------------------------------------ pointops (PAConv embedder, data side) ----
 * Op-level entry points for the reference's `pointops` kernels (models/scene_seg_PAConv/lib/pointops; python wrappers
 * lib/pointops/functions/pointops.py), point-major layouts, int32 indices, bit-exact INDICES against the reference's
 * compiled kernels (oracle/_ref/libpointops_ref.so, tests/test_pointops_gpu.py).
 *
 * fc_fps replaces `furthestsampling(xyz, m)` (pointops.py:47-62 -> src/sampling/sampling_cuda_kernel.cu:58-209):
 * xyz [B,n,3] -> idx_out [B,m] (first pick = point 0, then repeatedly the point farthest from the picked set);
 * new_xyz_out [B,m,3] optional (the gathered coordinates, `gathering` :68-90).  tie_block selects how equal
 * distances are resolved: 0 = exactly as the reference's launch does (its block of 2^floor(log2 n) <= 1024 threads
 * prefers the lowest thread, point k living in thread k % block), > 0 = that rule for an explicit block size,
 * < 0 = lowest index.  n <= 32768.  Also serves the data-side sub-sampling of the clouds
 * (dataloaders/ams_voxel_loader.py:298-307 uses torch_cluster.fps; same greedy rule, see DESIGN.md).              */
FC_API int fc_fps(const float* xyz, int B, int n, int m, int tie_block, int32_t* idx_out, float* new_xyz_out,
           fc_stream_t stream);

/* fc_knn_heap replaces `knnquery_heap(nsample, xyz, new_xyz)` (pointops.py:475-497 ->
 * src/knnquery_heap/knnquery_heap_cuda_kernel.cu:53-110): for each of the m queries the k nearest of the n points,
 * ascending squared distance; idx_out [B,m,k]; dist2_out [B,m,k] optional.  The reference's heap algorithm is followed
 * step for step (the order of exactly equal distances is an artefact of it; k > n leaves index 0 / 1e10 in the unfilled
 * slots).  1 <= k <= 40.                                                                                             */
FC_API int fc_knn_heap(const float* xyz, const float* new_xyz, int B, int n, int m, int k, int32_t* idx_out,
                float* dist2_out, fc_stream_t stream);

/* fc_three_nn replaces `nearestneighbor(unknown, known)` (pointops.py:96-115 ->
 * src/interpolation/interpolation_cuda_kernel.cu:134-213): unknown [B,n,3], known [B,m,3] -> the three nearest known
 * points of every unknown point: dist2_out [B,n,3] SQUARED distances (the python wrapper takes the sqrt), idx_out [B,n,3];
 * ties by lower index; m < 3 leaves index 0 / +inf in the unfilled slots.                                           */
FC_API int fc_three_nn(const float* unknown, const float* known, int B, int n, int m, float* dist2_out,
                int32_t* idx_out, fc_stream_t stream);

/* fc_three_interpolate replaces `interpolation(features, idx, weight)` (pointops.py:121-140 -> interpolation_cuda_kernel.cu:
 * 181-229) in point-major layout: known_feat [B,m,ldk] (C columns used), idx / weight [B,n,3] -> out [B,n,ldo]:
 * out = fma(w2, f[idx2], fma(w1, f[idx1], w0 * f[idx0])) (the contraction nvcc applies to the reference expression).  */
FC_API int fc_three_interpolate(const float* known_feat, int ldk, int C, const int32_t* idx, const float* weight,
                         int B, int n, int m, float* out, int ldo, fc_stream_t stream);

/* fc_group_points replaces `grouping(features, idx)` (pointops.py:158-175 -> src/grouping/grouping_cuda_kernel.cu:60-95) in
 * point-major layout: feat [B,n,ldf] (C columns), idx [B,m,k] -> out [B,m,k,ldo].                                      */
FC_API int fc_group_points(const float* feat, int ldf, int C, const int32_t* idx, int B, int n, int m, int k,
                    float* out, int ldo, fc_stream_t stream);

/* ------------------------------------------------------------------ GEMM (test hook) ------
 * C[M,N] = act(A[M,K] * Wt[K,N] + bias) with the library's fp32 GEMM; `Wt` is K-major
 * ([Kp, ldw], Kp = K rounded up to 16, rows >= K zero, ldw >= N rounded up to 128 (64 if N<=64)).
 * act: 0 none, 1 exact-erf GELU (reference models/nets.py:19-30 with nn.GELU), 2 LeakyReLU(0.2)
 * (reference models/pytorch_gcn.py:63-77).  precision: 0 = fp32 FFMA, 1 = 3xTF32 tcgen05.      */
FC_API int fc_gemm(const float* A, int lda, const float* Wt, int ldw, const float* bias,
            float* C, int ldc, int M, int N, int K, int act, int precision, fc_stream_t stream);

/* The same product on the tensor cores (3xTF32 tcgen05.mma, TMEM accumulators, TMA-fed): Whi / Wlo are
 * the TF32 hi / lo parts of W, N-major [ceil(N/192)*BN][ldk] with BN = ceil(N / ceil(N/192)) rounded up to
 * 16 and ldk = K rounded up to 32 (zero padded); A is split on chip.  Requires lda % 4 == 0, N >= 16.    */
FC_API int fc_gemm_tf32x3(const float* A, int lda, const float* Whi, const float* Wlo, int ldk,
                   const float* bias, float* C, int ldc, int M, int N, int K, int act, fc_stream_t stream);

/* Same product as 3xFP16: Whi16 = fp16(W), Wlo16 = fp16((W - Whi16) * 2^11), same [rows][ldk] layout with 2-byte
 * elements.  fp16 carries the same 11-bit significand as TF32, so the three products A_hi W_hi + 2^-11 (A_lo' W_hi +
 * A_hi W_lo') are as accurate as the TF32 ones at twice the tensor rate and half the operand bytes; the price is fp16's
 * exponent range: an activation with |a| >= 65520 turns its output row into NaN (loud, never a silently wrong value). */
FC_API int fc_gemm_f16x3(const float* A, int lda, const void* Whi16, const void* Wlo16, int ldk,
                  const float* bias, float* C, int ldc, int M, int N, int K, int act, fc_stream_t stream);

/* ------------------------------------------------------------------ EdgeConv --------------
 * One DGCNN EdgeConv block, reference models/pytorch_gcn.py:23-47 + :63-74 + :86-100:
 *   out_i = max_{j in idx_i} LeakyReLU_0.2( BN_eval( W * [x_j - x_i ; x_i] ) )
 * computed in the factorised form out_i = LeakyReLU( max_j P_j + Q_i ), P = x*(a.W1)^T,
 * Q = x*(a.(W2-W1))^T + b  (a, b = folded eval-mode BN).
 * PQ is [B*N, ldpq] with P in columns [0,Cout) and Q in [Cout, 2Cout) (produced by fc_gemm);
 * idx [B,N,k] int32 local indices; out [B*N, ldo] written at column 0..Cout-1.               */
FC_API int fc_edgeconv_gather_max(const float* PQ, int ldpq, const int32_t* idx, int B, int N, int k,
                           int Cout, float* out, int ldo, fc_stream_t stream);

/* ------------------------------------------------------------------ cross attention -------
 * softmax(q k^T * scale) v, single head, reference models/perceiver.py:108-115.
 * q [B*N, ldq] (dim d), kv [B*Nc, ldkv] with k in columns [0,d) and v in [d,2d); out [B*N, ldo].
 * Only d == 64 is supported.                                                                  */
FC_API int fc_cross_attention(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo,
                       int B, int N, int Nc, int d, float scale, fc_stream_t stream);

/* Same product on the tensor cores with warp-level MMA (mma.sync 3xTF32, flash style).                  */
FC_API int fc_cross_attention_tf32x3(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo,
                              int B, int N, int Nc, int d, float scale, fc_stream_t stream);

/* Same product on the 5th-gen tensor cores (tcgen05 + TMEM); the one the flow uses when precision = 1: 3xTF32 operands
 * (fc_cross_attention_tc, models packed with TF32 copies) or 3xFP16 operands (fc_cross_attention_tc_f16, models packed with
 * fp16 copies: half the operand bytes, twice the tensor rate).  Needs caller-provided device scratch (hi/lo copies of k and
 * of v transposed), 128-byte aligned.                                                                              */
FC_API int64_t fc_cross_attention_tc_scratch_bytes(int B, int Nc);
FC_API int fc_cross_attention_tc(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo,
                          int B, int N, int Nc, int d, float scale, void* scratch, int64_t scratch_bytes,
                          fc_stream_t stream);
FC_API int fc_cross_attention_tc_f16(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo,
                              int B, int N, int Nc, int d, float scale, void* scratch, int64_t scratch_bytes,
                              fc_stream_t stream);

/* The softmax weights of the same product, P = softmax(q k^T * scale) over the keys, written out (the flash kernels above never
 * form them): out [B, n_query, Nc], out[b, r, j] for query row query_idx[r] of cloud b (q row b*N + query_idx[r]; query_idx a
 * device int32 list, the same for every cloud, or NULL for all N rows with n_query == N).  Exact fp32: the dot product is a
 * sequential fma chain over the d = 64 dimensions, so every weight is deterministic and independent of the batch and of the
 * query list.  The kernel fc_flow_attention_maps runs per captured block.                                              */
FC_API int fc_attention_maps(const float* q, int ldq, const float* kv, int ldkv, const int32_t* query_idx, int n_query,
                      float* out, int B, int N, int Nc, float scale, fc_stream_t stream);

/* ------------------------------------------------------------------ data-side ops ----------
 * What the reference's loader does between reading a voxel and calling `inner_loop` (SURVEY.md 8f rank 4).
 * fc_fps_points replaces `voxel[fps(voxel, batch, ratio=n_samples/len(voxel), random_start=False)][:n_samples]`
 * (reference dataloaders/ams_voxel_loader.py:298-307; torch_cluster.fps): furthest point sampling over ALL C point
 * columns (C = 3 or 6), first pick = point 0, ties to the lowest index.  pts [B][n][ld]; idx_out [B][m];
 * pts_out [B][m][ld_out] (first C columns written) or NULL.
 * fc_co_unit_sphere replaces `co_unit_sphere(points_0, points_1, return_inverse=True)` (reference utils.py:259-280,
 * called by ams_voxel_loader.py:357-358): the xyz columns of both clouds of a pair are shifted by their JOINT mean and
 * divided by the largest norm, in place; inverse_out [B][4] = (mean xyz, furthest_distance) or NULL.            */
FC_API int fc_fps_points(const float* pts, int ld, int B, int n, int C, int m, int32_t* idx_out, float* pts_out,
                  int ld_out, fc_stream_t stream);
FC_API int fc_co_unit_sphere(float* points_0, int n0, int ld0, float* points_1, int n1, int ld1, int B,
                      float* inverse_out, fc_stream_t stream);

/* ------------------------------------------------------------------ model handles ---------
 * A model is described by (header int32[], table int64[], arena fp32[] on the device), produced by
 * flowcompare_b200/packing.py from the reference's own `state_dict`s (SURVEY.md A.5).  The arena
 * stays owned by the caller and must outlive the handle.  See DESIGN.md "arena format".       */
typedef struct fc_flow fc_flow;
typedef struct fc_embedder fc_embedder;

FC_API int fc_flow_create(const int32_t* header_host, int n_header, const int64_t* table_host, int n_table,
                   const float* arena, int64_t arena_floats, fc_flow** out);
FC_API void fc_flow_destroy(fc_flow* h);
FC_API int64_t fc_flow_workspace_bytes(const fc_flow* h, int B, int N, int Nc);
/* fc_flow_log_prob replaces `Flow.log_prob(x, context, extra_context)`, reference
 * models/transform.py:70-76, for the transform list built by model_initialization.py:134-152.
 *   x [B,N,input_dim]; context [B,Nc,E] (attention configs) or [B,E] (global embedder);
 *   extra [B] or NULL; eps [B,N,latent-input_dim] = the N(0,1) draw of
 *   models/distributions.py:148-153 made explicit; log_prob_out [B,N].
 *   precision: 0 = fp32 FFMA GEMMs, 1 = tcgen05 GEMMs (3xTF32 or 3xFP16, whichever weight
 *   copies the model was packed with).                                                        */
FC_API int fc_flow_log_prob(const fc_flow* h, const float* x, const float* context, const float* extra,
                     const float* eps, float* log_prob_out, int B, int N, int Nc,
                     void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream);

/* Flows built from the transforms no shipped config selects (reference model_initialization.py:95-131): the packed model
 * says which coupling it carries -- `RationalQuadraticSplineCoupling.forward` (models/spline_coupling.py:187-210 over
 * :24-169), `ExponentialCoupling.forward` (models/exponential_coupling.py:44-58) -- which permuter (`Permuter`,
 * `FullCombiner`, `ExponentialCombiner`, models/permuters.py:15-66, folded with ActNorm into the same 300x300 GEMM as
 * LinearLU), ReLU conditioners, and the identity augmenter (latent_dim == input_dim: pass eps = NULL); fc_flow_log_prob
 * runs all of them.  `CIFblock.forward` (models/cif_block.py:71-100: `Augment`, `Reverse`, `AffineCoupling`, ActNorm,
 * `Reverse`, `Slice` of models/slice.py:31-44, then the coupling) draws noise of its own in every block, so flows with
 * latent_dim < cif_latent_dim go through fc_flow_log_prob_cif: eps_cif [L, B, N, fc_flow_cif_noise_dim(h)] holds the
 * blocks' N(0,1) draws in transform-list order.                                                                  */
FC_API int fc_flow_log_prob_cif(const fc_flow* h, const float* x, const float* context, const float* extra,
                         const float* eps, const float* eps_cif, float* log_prob_out, int B, int N, int Nc,
                         void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream);
FC_API int fc_flow_cif_noise_dim(const fc_flow* h);

/* Multi-draw log-likelihood.  A log-prob is a single-sample estimate of log p(x | c): the augmenter's noise dims are drawn from
 * q(e | x, c) (reference models/augmenter.py:49-63) and every CIF block draws again.  fc_flow_log_prob_draws scores K draws per
 * point in one pass: the augmenter's network runs once per point, only its output layer once per draw, and the coupling layers
 * see K*N points per cloud (the context's to_kv runs once per layer per cloud, not per draw).
 *   eps [K, B, N, latent-input_dim] (NULL for an identity augmenter); eps_cif [L, B, K, N, fc_flow_cif_noise_dim(h)] (draw k of
 *   cloud b at eps_cif[l][b][k]; NULL for flows without CIF blocks); lp_draws_out [K, B, N].  The rest as fc_flow_log_prob_cif.
 *   lp_draws_out[k] is bitwise what fc_flow_log_prob / fc_flow_log_prob_cif return for eps[k] and draw k's eps_cif.
 * One pass runs at most 2^20 rows: K*B*N <= 2^20 (B*N for a flow with no stochastic transform -- identity augmenter and no
 * CIF block -- which is evaluated once and its log-prob copied to the K slots), else FC_ERR_INVALID_ARG; callers split the
 * draws over several passes.  fc_flow_log_prob_draws_workspace_bytes(h, B, N, Nc, K) sizes the workspace (FC_ERR_WORKSPACE if
 * it is smaller).                                                                                                          */
FC_API int64_t fc_flow_log_prob_draws_workspace_bytes(const fc_flow* h, int B, int N, int Nc, int K);
FC_API int fc_flow_log_prob_draws(const fc_flow* h, const float* x, const float* context, const float* extra,
                           const float* eps, const float* eps_cif, int K, float* lp_draws_out, int B, int N, int Nc,
                           void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream);

/* The importance-weighted estimate over the leading axis: out[i] = log((1/K) sum_k exp(draws[k][i])) for draws [K, M], as
 * m + (log(sum_k exp(draws[k][i] - m)) - log K), m = max_k draws[k][i], in fp32 with the draws folded in index order -- so the
 * result depends on the point's K values only, not on M or on how the draws were split over passes.  Any NaN draw gives NaN,
 * any +inf draw +inf; -inf draws drop out of the sum, all -inf gives -inf.  K equal finite draws give that value exactly.
 * A caller that splits the draws over several fc_flow_log_prob_draws passes reduces once at the end.                     */
FC_API int fc_logmeanexp(const float* draws, int K, int64_t M, float* out, fc_stream_t stream);

/* Op-level entry points of the two couplings' elementwise tails (the conditioner MLP is a chain of fc_gemm calls).
 * fc_rq_spline replaces `unconstrained_rational_quadratic_spline(inputs, unnormalized_widths, unnormalized_heights,
 * unnormalized_derivatives, inverse)` (reference models/spline_coupling.py:24-66 over :69-169; 'linear' tails, tail bound 3,
 * num_bins <= 16): params [M][ldp], element j's (3*num_bins+1) values contiguous as [widths | heights | derivatives] (the
 * reshape + split of :197-198); x [M][ldx], n elements per row, transformed in place; forward ADDS the row's summed
 * log|det| to logabsdet_rowsum[row] (zero it first), inverse ignores it.
 * fc_expm_action replaces the x2 update of `ExponentialCoupling.forward / .inverse` (reference
 * models/exponential_coupling.py:48-58, :68-77): params [M][ldp] = [w n*n | b n] per row, squash4 = device pointer to
 * (scale, shift, rescale, reshift); forward x <- expm(W) x + b and trace_rowsum[row] += trace W, inverse
 * x <- expm(-W)(x - b); n <= 256.  expm(W) is never formed: its action on the vector is computed.               */
FC_API int fc_rq_spline(const float* params, int ldp, float* x, int ldx, int n, int num_bins, int M,
                 float* logabsdet_rowsum, int inverse, fc_stream_t stream);
FC_API int fc_expm_action(const float* params, int ldp, float* x, int ldx, int n, const float* squash4,
                   float* trace_rowsum, int M, int inverse, fc_stream_t stream);

/* Same pass, additionally returning the final latent z_out [B,N,latent] (the point of the base density; the input of
 * the sampling pass run backwards).                                                                              */
FC_API int fc_flow_forward(const fc_flow* h, const float* x, const float* context, const float* extra,
                    const float* eps, float* log_prob_out, float* z_out, int B, int N, int Nc,
                    void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream);

/* The same forward pass, additionally writing the cross-attention weights of chosen attention blocks: the
 * softmax(q k^T * 64^-1/2) over the context points of reference models/perceiver.py:108-115, which the flash kernels never form.
 * Slot 0 is the augmenter's attention (transforms.0.attn), slot l+1 coupling layer l's pre-conditioner attention.
 *   slots_host [n_slots]: HOST array, strictly increasing, each in [0, n_flow_layers]; query_idx [n_query]: device int32 rows of
 *   x (the same for every cloud, repeats allowed, each in [0, N): the caller's contract) or NULL for all N rows (n_query == N);
 *   maps_out [n_slots, B, n_query, Nc]: maps_out[i, b, r, j] = weight of context point j for query row query_idx[r] of cloud b in
 *   block slots_host[i]; rows sum to 1.  The rest as fc_flow_log_prob_cif (eps_cif NULL for flows without CIF blocks);
 *   log_prob_out is bitwise what fc_flow_log_prob returns.  fc_flow_workspace_bytes(h, B, N, Nc) sizes the workspace.
 * FC_ERR_INVALID_ARG for slot 0 of a flow with an identity augmenter, unsorted or out-of-range slots, or query_idx == NULL with
 * n_query != N; FC_ERR_UNSUPPORTED for global-embedding flows (their conditioners attend to no context points).          */
FC_API int fc_flow_attention_maps(const fc_flow* h, const float* x, const float* context, const float* extra, const float* eps,
                           const float* eps_cif, const int32_t* slots_host, int n_slots, const int32_t* query_idx, int n_query,
                           float* maps_out, float* log_prob_out, int B, int N, int Nc, void* workspace,
                           int64_t workspace_bytes, int precision, fc_stream_t stream);

/* Inverse / sampling pass: fc_flow_sample replaces `Flow.sample` after its base draw (reference models/transform.py:79-84,
 * called by `make_sample`, model_initialization.py:231-245): the transforms walked backwards with each `.inverse`
 * (models/affine_coupling.py:48-62, models/permuters.py:171-177, models/act_norm.py:45-46, models/augmenter.py:20-21,65-67).
 *   z [B,P,latent] the base draw (reference: sample_dist.sample = N(loc, scale), P = n_points); context / extra as in
 *   fc_flow_log_prob; x_out [B,P,input_dim].  fc_flow_workspace_bytes(h, B, P, Nc) sizes the workspace.
 * The inverse ActNorm+LinearLU matrices are not part of the forward model: fc_flow_set_inverse attaches them first
 * (header/table/arena from packing.pack_flow_inverse; the arena must outlive the handle); without it fc_flow_sample
 * returns FC_ERR_MODEL.                                                                                          */
FC_API int fc_flow_set_inverse(fc_flow* h, const int32_t* header_host, int n_header, const int64_t* table_host,
                        int n_table, const float* arena, int64_t arena_floats);
FC_API int fc_flow_sample(const fc_flow* h, const float* z, const float* context, const float* extra, float* x_out,
                   int B, int P, int Nc, void* workspace, int64_t workspace_bytes, int precision,
                   fc_stream_t stream);
/* The same pass for flows with CIF blocks (`CIFblock.inverse`, reference models/cif_block.py:102-111): every block's
 * `Slice.inverse` SAMPLES the columns that were sliced off (models/slice.py:46-58); eps_cif [L, B, P, fc_flow_cif_noise_dim(h)]
 * holds those N(0,1) draws, indexed by the block's position in the forward list.  fc_flow_sample itself covers every other
 * flow: the three couplings' inverses (models/affine_coupling.py:48-62, models/spline_coupling.py:212-227,
 * models/exponential_coupling.py:60-77) and every permuter's (models/permuters.py:22-26, :51-53, :67-69, :171-177).      */
FC_API int fc_flow_sample_cif(const fc_flow* h, const float* z, const float* context, const float* extra,
                       const float* eps_cif, float* x_out, int B, int P, int Nc, void* workspace,
                       int64_t workspace_bytes, int precision, fc_stream_t stream);

/* Input gradients: what autograd of `Flow.log_prob` (reference models/transform.py:70-76) gives with respect to the target
 * points, `torch.autograd.grad(flow.log_prob(x, context=...).sum(), x)` with the augmentation noise eps held fixed.  A point's
 * log-prob depends on that point and the context only, so grad_out[b, n, :] = d log_prob[b, n] / d x[b, n, :input_dim] is the
 * whole Jacobian.  The context, the extra context and the weights are constants (no gradient flows to them).
 *   fc_flow_set_grad attaches the transposed weights the backward GEMMs run (header/table/arena from packing.pack_flow_grad, always
 *   3xTF32 tensor-core copies; the arena must outlive the handle); without it fc_flow_log_prob_grad returns FC_ERR_MODEL.
 *   fc_flow_log_prob_grad: arguments as fc_flow_log_prob, plus grad_out [B, N, input_dim].  It runs the forward pass, keeping the
 *   latent at the input of every coupling layer, then walks the layers backwards, recomputing each layer's forward from its
 *   checkpoint.  log_prob_out is bitwise what fc_flow_log_prob returns.  Affine couplings only: flows with spline or exponential
 *   couplings or CIF blocks return FC_ERR_UNSUPPORTED.  fc_flow_log_prob_grad_workspace_bytes(h, B, N, Nc) sizes the workspace
 *   (about 181 KB per point at the shipped widths, most of it the checkpoints); one pass runs at most 2^16 points (B*N), else
 *   FC_ERR_INVALID_ARG.                                      */
FC_API int fc_flow_set_grad(fc_flow* h, const int32_t* header_host, int n_header, const int64_t* table_host, int n_table,
                     const float* arena, int64_t arena_floats);
FC_API int64_t fc_flow_log_prob_grad_workspace_bytes(const fc_flow* h, int B, int N, int Nc);
FC_API int fc_flow_log_prob_grad(const fc_flow* h, const float* x, const float* context, const float* extra, const float* eps,
                          float* log_prob_out, float* grad_out, int B, int N, int Nc, void* workspace,
                          int64_t workspace_bytes, int precision, fc_stream_t stream);

FC_API int fc_embedder_create(const int32_t* header_host, int n_header, const int64_t* table_host, int n_table,
                       const float* arena, int64_t arena_floats, fc_embedder** out);
FC_API void fc_embedder_destroy(fc_embedder* h);
FC_API int64_t fc_embedder_workspace_bytes(const fc_embedder* h, int B, int Nc);
/* fc_embed replaces `input_embedder(extract_0)`: DGCNNembedder.forward (reference
 * models/pytorch_gcn.py:81-107) -> out [B,Nc,E]; DGCNNembedderGlobal.forward (:143-188) -> out [B,E];
 * PointNet2SSGSeg.forward (models/scene_seg_PAConv/model/pointnet2/pointnet2_paconv_seg.py:63-82)
 * -> out [B,Nc,E].  pts [B,Nc,input_dim].  knn_idx_out: optional int32 [4,B,Nc,k] (DGCNN only).  */
FC_API int fc_embed(const fc_embedder* h, const float* pts, float* out, int B, int Nc,
             int32_t* knn_idx_out, void* workspace, int64_t workspace_bytes, int precision,
             fc_stream_t stream);

/* ------------------------------------------------------------------ whole path ------------
 * fc_inner_loop replaces `inner_loop(batch, models_dict, config)`, reference
 * model_initialization.py:206-228: embed extract_0, score extract_1.  Device buffers.
 * Outputs: log_prob_out [B,N]; stats_out[2] = {loss = -mean(log_prob), bpd = loss*log2(e)/input_dim}. */
FC_API int64_t fc_inner_loop_workspace_bytes(const fc_embedder* e, const fc_flow* f, int B, int N, int Nc);
FC_API int fc_inner_loop(const fc_embedder* e, const fc_flow* f, const float* extract_0, const float* extract_1,
                  const float* extra, const float* eps, float* log_prob_out, float* stats_out,
                  int B, int N, int Nc, void* workspace, int64_t workspace_bytes, int precision,
                  fc_stream_t stream);
/* Same call with HOST buffers (pinned or pageable): copies inputs H2D, runs, copies log_prob and
 * stats D2H on `stream`, and synchronises the stream before returning.  This is the call the
 * end-to-end benchmark times.  The staging area is carved from `workspace`.                    */
FC_API int64_t fc_inner_loop_host_workspace_bytes(const fc_embedder* e, const fc_flow* f, int B, int N, int Nc);
FC_API int fc_inner_loop_host(const fc_embedder* e, const fc_flow* f, const float* extract_0_host,
                       const float* extract_1_host, const float* extra_host, const float* eps_host,
                       float* log_prob_out_host, float* stats_out_host, int B, int N, int Nc,
                       void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream);

/* ------------------------------------------------------------------ consumers -------------
 * fc_change_score replaces `log_prob_to_change` + `clamp_infs`, reference test_flow.py:241-275:
 * +-inf entries are replaced by the minimum finite value OF THE WHOLE [B,N] TENSOR (what `clamp_infs` does; the inputs are
 * not modified, unlike the reference's in-place clamp), then per cloud: mask = lp10 < mean(lp00) - multiple*std(lp00)
 * (unbiased std) or lp10 < hard_cutoff when use_hard_cutoff != 0, change = 1-(lp10-min)/(max-min), zero outside the mask.
 * lp10, lp00, change_out: [B,N].                                                                */
FC_API int fc_change_score(const float* lp10, const float* lp00, float* change_out, int B, int N,
                    float multiple, int use_hard_cutoff, float hard_cutoff, fc_stream_t stream);

/* Standard-normal fill (Philox-4x32-10 + Box-Muller) for callers that do not inject eps.      */
FC_API int fc_fill_normal(float* out, int64_t n, uint64_t seed, uint64_t offset, fc_stream_t stream);

/* Per-class kernel timing for ONE instrumented step (bench.py's roofline): fc_profile_begin() makes every
 * launcher bracket its kernel with CUDA events; fc_profile_end() synchronises the device and returns, per
 * class (0 fp32 GEMM, 1 tcgen05 GEMM, 2 attention, 3 kNN, 4 EdgeConv gather-max, 5 other), the summed
 * milliseconds, algorithmic flops, algorithmic bytes and launch counts.  n_classes must be >= 6.        */
FC_API int fc_profile_begin(void);
FC_API int fc_profile_end(double* ms, double* flops, double* bytes, int64_t* launches, int n_classes);

/* Number of kernels this library has launched in this process since load (bench bookkeeping). */
FC_API int64_t fc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FLOWCOMPARE_B200_H */
