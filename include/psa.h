/*
 * psa.h -- C ABI of libpsa.so: the B200-native (sm_100a) point-set-abstraction hot path.
 *
 * This is the drop-in boundary.  The reference (hkust-vgd/scanobjectnn) reaches its native code through
 * plain C++ "Launcher" functions called from TensorFlow OpKernel::Compute (raw device pointers + int
 * dims, caller-owned buffers); every entry point below names the reference interface it replaces.
 * Reference paths are relative to pointnet2/tf_ops/ unless they start with dgcnn/ or pointnet2/.
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer to a dense, contiguous, row-major fp32 / int32 buffer owned by
 *     the caller; nothing is allocated or freed inside the library; outputs must not alias inputs;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream, which is what the
 *     reference's `<<<grid,block>>>` launches use); calls are asynchronous on that stream;
 *   - return value: PSA_OK (0); PSA_ERR_INVALID_ARGUMENT (-1) for a shape/attribute the reference's
 *     OP_REQUIRES would reject (message via psa_last_error()); PSA_ERR_UNSUPPORTED (-2) for a shape
 *     outside the compiled limits; a positive value is the cudaError_t of a failed launch.  Unlike the
 *     reference (which never checks), launches are checked with cudaGetLastError();
 *   - b == 0 or an empty extent is a successful no-op;
 *   - thread-safe: no global mutable state except the thread-local error string.
 */
#ifndef PSA_H_
#define PSA_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSA_OK 0
#define PSA_ERR_INVALID_ARGUMENT (-1)
#define PSA_ERR_UNSUPPORTED (-2)

typedef void* psa_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define PSA_API __attribute__((visibility("default")))
#else
#define PSA_API
#endif

/* library identity / diagnostics */
PSA_API int psa_version(void);                 /* MAJOR*10000 + MINOR*100 + PATCH */
PSA_API const char* psa_last_error(void);      /* thread-local, valid until the next failing call on this thread */
PSA_API int psa_sm_arch(void);                 /* 100: the only architecture compiled in (sm_100a) */

/* ---------------------------------------------------------------------------------------------
 * sampling/  (tf_sampling.cpp, tf_sampling_g.cu)
 * ------------------------------------------------------------------------------------------- */

/* Farthest point sampling.  Replaces
 *   void farthestpointsamplingLauncher(int b,int n,int m,const float* inp,float* temp,int* out)
 *   (sampling/tf_sampling.cpp:94, kernel tf_sampling_g.cu:105-170; op FarthestPointSample :28-40).
 * xyz (b,n,3) -> idx (b,m) int32; seed index 0; ties between equal maxima resolved exactly as the
 * reference's 512-thread strided scan + tree do: minimum over (k mod 512, k).  No `temp` scratch is
 * needed (running distances live in registers).  If new_xyz != NULL the gather of the sampled points
 * (GatherPoint, below) is fused: new_xyz (b,m,3).  Requires n >= 1 when m >= 1; m may exceed n. */
PSA_API int psa_farthest_point_sample(int b, int n, int m, const float* xyz, int* idx, float* new_xyz,
                              psa_stream_t stream);

/* Replaces gatherpointLauncher (sampling/tf_sampling.cpp:125, tf_sampling_g.cu:172-181).
 * inp (b,n,3), idx (b,m) -> out (b,m,3). */
PSA_API int psa_gather_point(int b, int n, int m, const float* inp, const int* idx, float* out, psa_stream_t stream);

/* Replaces cudaMemset + scatteraddpointLauncher (sampling/tf_sampling.cpp:150,174; tf_sampling_g.cu:183-192).
 * out_g (b,m,3), idx (b,m) -> inp_g (b,n,3), every element written.  Ordered (no float atomics): see
 * psa_scatter_workspace_bytes(b, n, m). */
PSA_API int psa_gather_point_grad(int b, int n, int m, const float* out_g, const int* idx, float* inp_g, void* workspace,
                          size_t workspace_bytes, psa_stream_t stream);

/* The three scatter-add gradients (GatherPointGrad, GroupPointGrad, ThreeInterpolateGrad) add the contributions of one
 * destination in ascending entry order -- the order of the reference's sequential CPU loops (grouping/test/ ..._cpu, tf_interpolate.cpp)
 * -- instead of the float atomicAdd of its CUDA kernels: results are bit-reproducible.  They need a device scratch buffer of
 * this many bytes for the per-cloud (destination -> entries) lists: b clouds, n_dst destination points and `entries`
 * scattered rows per cloud (m; m*nsample; 3*n).  Out-of-range indices are dropped.  n_dst <= 51200. */
PSA_API size_t psa_scatter_workspace_bytes(int b, int n_dst, long long entries);

/* ---------------------------------------------------------------------------------------------
 * grouping/  (tf_grouping.cpp, tf_grouping_g.cu)
 * ------------------------------------------------------------------------------------------- */

/* Replaces queryBallPointLauncher (grouping/tf_grouping.cpp:66, tf_grouping_g.cu:3-36; op QueryBallPoint :13-30).
 * xyz1 (b,n,3) dataset, xyz2 (b,m,3) queries -> idx (b,m,nsample), pts_cnt (b,m).
 * First `nsample` points in index order with max(sqrtf(d2),1e-20f) < radius; unused slots repeat the
 * first hit.  A query with an empty ball gets idx row = 0 and pts_cnt = 0 (the reference leaves that
 * row uninitialised).  pts_cnt may be NULL. */
PSA_API int psa_query_ball_point(int b, int n, int m, float radius, int nsample, const float* xyz1, const float* xyz2,
                         int* idx, int* pts_cnt, psa_stream_t stream);

/* Replaces groupPointLauncher (grouping/tf_grouping.cpp:142, tf_grouping_g.cu:40-57).
 * points (b,n,c), idx (b,m,nsample) -> out (b,m,nsample,c). */
PSA_API int psa_group_point(int b, int n, int c, int m, int nsample, const float* points, const int* idx, float* out,
                    psa_stream_t stream);

/* Replaces cudaMemset + groupPointGradLauncher (grouping/tf_grouping.cpp:173,204; tf_grouping_g.cu:61-78).
 * grad_out (b,m,nsample,c), idx -> grad_points (b,n,c), every element written.
 * workspace: psa_scatter_workspace_bytes(b, n, m*nsample). */
PSA_API int psa_group_point_grad(int b, int n, int c, int m, int nsample, const float* grad_out, const int* idx,
                         float* grad_points, void* workspace, size_t workspace_bytes, psa_stream_t stream);

/* Replaces selectionSortLauncher (grouping/tf_grouping.cpp:108, tf_grouping_g.cu:83-123; op SelectionSort).
 * dist (b,m,n) -> outi (b,m,n) int32, out (b,m,n): full copies whose first k slots per row hold the k
 * smallest, produced by the reference's swap-based partial selection sort (ties by current position). */
PSA_API int psa_selection_sort(int b, int n, int m, int k, const float* dist, int* outi, float* out, psa_stream_t stream);

/* knn_point (grouping/tf_grouping.py:49-74) without the (b,m,n) matrices: xyz1 (b,n,c) dataset,
 * xyz2 (b,m,c) queries -> val (b,m,k), idx (b,m,k); same distances (sum_c (a-b)^2, sequential,
 * un-contracted) and the same swap-based tie order as SelectionSort. */
PSA_API int psa_knn_point(int b, int n, int m, int c, int k, const float* xyz1, const float* xyz2, float* val, int* idx,
                  psa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * 3d_interpolation/  (tf_interpolate.cpp -- CPU-only ops in the reference)
 * ------------------------------------------------------------------------------------------- */

/* Replaces threenn_cpu (3d_interpolation/tf_interpolate.cpp:60-103; op ThreeNN :12-21).
 * xyz1 (b,n,3) unknown, xyz2 (b,m,3) known -> dist (b,n,3) SQUARED distances ascending, idx (b,n,3).
 * Strict-< cascade (earlier k wins ties); slots beyond m are dist=+inf, idx=0. */
PSA_API int psa_three_nn(int b, int n, int m, const float* xyz1, const float* xyz2, float* dist, int* idx,
                 psa_stream_t stream);

/* Replaces threeinterpolate_cpu (tf_interpolate.cpp:107-127).
 * points (b,m,c), idx (b,n,3), weight (b,n,3) -> out (b,n,c) = (p1*w1 + p2*w2) + p3*w3. */
PSA_API int psa_three_interpolate(int b, int m, int c, int n, const float* points, const int* idx, const float* weight,
                          float* out, psa_stream_t stream);

/* Replaces memset + threeinterpolate_grad_cpu (tf_interpolate.cpp:131-153,258).
 * grad_out (b,n,c), idx, weight -> grad_points (b,m,c), every element written; bit-identical to the reference's CPU loop
 * (same order, product rounded before the add).  workspace: psa_scatter_workspace_bytes(b, m, 3*n). */
PSA_API int psa_three_interpolate_grad(int b, int n, int c, int m, const float* grad_out, const int* idx,
                               const float* weight, float* grad_points, void* workspace, size_t workspace_bytes,
                               psa_stream_t stream);

/* The interpolation half of pointnet_fp_module (pointnet2/utils/pointnet_util.py:211-216) in one launch:
 * three_nn -> dist=max(dist,1e-10) -> w=(1/dist)/sum(1/dist) -> three_interpolate.
 * Optional outputs dist/idx/weight (b,n,3) may be NULL. */
PSA_API int psa_three_nn_interpolate(int b, int n, int m, int c, const float* xyz1, const float* xyz2,
                             const float* points2, float* out, float* dist, int* idx, float* weight,
                             psa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * input pipeline  (data_utils.py:133-186, pointnet2/utils/provider.py:34-52,189-236, train.py:246-252 -- numpy on the
 * host in the reference, one kernel here).  src (b,n_src,3) -> out (b,n,3):
 *   [center over all n_src points] -> [divide by the max norm] -> gather perm[0..n) (same subset for every cloud; NULL =
 *   the first n points) -> [dropout: dropped points := the cloud's first batch point] -> [rotate about the up axis by
 *   (cos,sin) given in double, float64 product] -> [scale (b)] -> [shift (b,3)] -> [+ clip(sigma * noise, -clip, clip),
 *   float64 sum].  Every optional input may be NULL (step skipped).  The random numbers are inputs; see ops.augment_batch.
 * ------------------------------------------------------------------------------------------- */
PSA_API int psa_augment_batch(int b, int n_src, int n, const float* src, const int* perm, const double* cos_sin,
                              const float* scale, const float* shift, const float* noise, double sigma, double clip,
                              const unsigned char* drop, int center, int normalize, float* out, psa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * dgcnn graph functions  (dgcnn/utils/tf_util.py:638-706 -- TF library ops in the reference)
 * ------------------------------------------------------------------------------------------- */

/* pairwise_distance (dgcnn/utils/tf_util.py:638-657): x (b,n,c) -> adj (b,n,n),
 * adj = (|x_i|^2 + (-2 x_i.x_j)) + |x_j|^2 with fma chains over c (canonical order, oracle/psa_oracle.c). */
PSA_API int psa_pairwise_distance(int b, int n, int c, const float* x, float* adj, psa_stream_t stream);

/* knn (dgcnn/utils/tf_util.py:660-671): adj (b,n,ncols) -> nn_idx (b,n,k): top_k(-adj), ascending adj,
 * lower index first on ties. */
PSA_API int psa_knn_topk(int b, int n, int ncols, int k, const float* adj, int* nn_idx, psa_stream_t stream);

/* pairwise_distance + knn fused, never materialising (b,n,n): x (b,n,c) -> nn_idx (b,n,k). */
PSA_API int psa_knn_graph(int b, int n, int c, int k, const float* x, int* nn_idx, psa_stream_t stream);

/* get_edge_feature (dgcnn/utils/tf_util.py:674-706): x (b,n,c), nn_idx (b,n,k) -> (b,n,k,2c) = [x_i, x_j-x_i]. */
PSA_API int psa_get_edge_feature(int b, int n, int c, int k, const float* x, const int* nn_idx, float* out,
                         psa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * grouped shared MLP  (pointnet2/utils/pointnet_util.py:87-154, tf_util.conv2d 1x1 + BN + ReLU,
 * dgcnn EdgeConv dgcnn/models/dgcnn.py:31-80) -- TF/cuDNN library ops in the reference
 * ------------------------------------------------------------------------------------------- */

/* One per-row shared MLP: up to PSA_MAX_MLP_LAYERS layers of  y = relu?( (x . W) * scale + shift ).
 *   channels[0..n_layers]   C_0 (input) ... C_L
 *   weight[l]  (C_l, C_{l+1}) row-major  == TF conv kernel (1,1,C_in,C_out) (tf_util.py:162-168)
 *   scale[l], shift[l]  (C_{l+1}): conv bias + inference-mode batch norm folded by the caller:
 *        scale = gamma / sqrt(moving_var + 1e-3),  shift = (bias - moving_mean) * scale + beta
 *        (no BN: scale = 1, shift = bias);  scale[l] may be NULL (= all ones)
 *   relu[l]    nonzero -> ReLU after layer l */
#define PSA_MAX_MLP_LAYERS 4
typedef struct psa_mlp {
    int n_layers;
    int channels[PSA_MAX_MLP_LAYERS + 1];
    const float* weight[PSA_MAX_MLP_LAYERS];
    const float* scale[PSA_MAX_MLP_LAYERS];
    const float* shift[PSA_MAX_MLP_LAYERS];
    int relu[PSA_MAX_MLP_LAYERS];
    /* Optional, for weights that do not change between calls (inference): tensor-core weight images built ONCE by
     * psa_prepare_weight_image().  image[l] == NULL -> the entry point builds the image in its workspace on every call
     * (~45 us per PointNet++ forward).  An image is only used if its tile width / first row match what the entry point
     * needs (psa_mlp_image_plan() tells); otherwise it is ignored and rebuilt. */
    const void* image[PSA_MAX_MLP_LAYERS];
    int image_nt[PSA_MAX_MLP_LAYERS];      /* tile width the image was built for, as returned by psa_mlp_image_plan (64 or 128, | 0x200 = fp16x2 blocks followed by their bf16x3 twin, | 0x100 = bf16x3 only) */
    int image_row0[PSA_MAX_MLP_LAYERS];    /* first row of weight[l] covered by the image (3 when the xyz rows are split off) */
} psa_mlp;

/* Which images would an entry point use for this MLP?  usage: 0 = psa_shared_mlp(rows, pool_k), 1 = psa_sa_group_all_infer
 * (rows = b*n, c), 2 = psa_sa_module_infer (rows = b*n, c, nsample).  Fills nt/row0/bytes per layer (bytes 0 = that layer
 * does not run on the tensor cores).  Returns PSA_OK. */
#define PSA_USAGE_SHARED_MLP 0
#define PSA_USAGE_SA_GROUP_ALL 1
#define PSA_USAGE_SA_MODULE 2
PSA_API int psa_mlp_image_plan(int usage, long long rows, int pool_k, int c, int nsample, const psa_mlp* mlp,
                               int nt[PSA_MAX_MLP_LAYERS], int row0[PSA_MAX_MLP_LAYERS], size_t bytes[PSA_MAX_MLP_LAYERS]);
/* Build the image of rows [row0, K) of W (K, N) for tile width | format `nt` into `image` (bytes from psa_mlp_image_plan).
 * An fp16x2 image is followed, in the same buffer, by the bf16x3 image the range guard reruns on. */
PSA_API int psa_prepare_weight_image(int K, int N, int row0, int nt, const float* W, void* image, psa_stream_t stream);

/* Dense rows: x (rows, C_0) -> out.  pool_k == 1: out (rows, C_L).  pool_k > 1: rows must be a multiple
 * of pool_k and out (rows/pool_k, C_L) = channel-wise max over each run of pool_k consecutive rows
 * (tf.reduce_max over nsample, pointnet_util.py:127); pool_k must divide 128 (>= 8) or be a multiple of 128.
 * Used for sample_and_group_all (SA3), FP-module convs, DGCNN's point-wise convs and the FC heads.
 * Layers run one launch each; the (rows, C_l) intermediates ping-pong through the caller's workspace of
 * psa_shared_mlp_workspace_bytes(rows, mlp) bytes (0 for a single layer; workspace may then be NULL). */
PSA_API size_t psa_shared_mlp_workspace_bytes(long long rows, const psa_mlp* mlp);
PSA_API int psa_shared_mlp(long long rows, int pool_k, const float* x, const psa_mlp* mlp, float* out,
                           void* workspace, size_t workspace_bytes, psa_stream_t stream);

/* Fused set-abstraction level, inference mode (pointnet_sa_module, pointnet_util.py:87-154 with
 * sample_and_group :22-56 inside): for every query j of new_xyz
 *   idx_j  = query_ball_point(radius, nsample, xyz, new_xyz)[j]           (or caller-provided idx)
 *   row_k  = [ xyz[idx_jk] - new_xyz[j]  ,  points[idx_jk] ]               (xyz first, :46-50)
 *   out_j  = max_k  MLP(row_k)
 * without materialising the (b,m,nsample,3+c) tensor.  xyz (b,n,3), new_xyz (b,m,3), points (b,n,c) or
 * NULL with c = 0, mlp->channels[0] must equal 3 + c.  out (b,m,C_L).
 * idx_in  != NULL: use these neighbourhoods (b,m,nsample) instead of searching;
 * idx_out != NULL / pts_cnt != NULL: also write the ball-query result (idx_out is REQUIRED when idx_in is NULL).
 * workspace: psa_sa_module_workspace_bytes() bytes of device scratch (per-point layer-1 products), may be 0/NULL. */
PSA_API size_t psa_sa_module_workspace_bytes(int b, int n, int m, int c, int nsample, const psa_mlp* mlp);
PSA_API int psa_sa_module_infer(int b, int n, int m, int c, float radius, int nsample, const float* xyz,
                                const float* new_xyz, const float* points, const int* idx_in, const psa_mlp* mlp,
                                float* out, int* idx_out, int* pts_cnt, void* workspace, size_t workspace_bytes,
                                psa_stream_t stream);

/* pointnet_sa_module with group_all=True (pointnet_util.py:59-84,113-127): rows [xyz, points] (xyz first) -> MLP -> max over
 * the n points of each cloud, without building the (b,n,3+c) concatenation.  xyz (b,n,3), points (b,n,c), mlp->channels[0]
 * == 3 + c -> out (b, C_L).  Returns PSA_ERR_UNSUPPORTED when the first layer cannot run on the tensor-core path (then
 * concatenate and call psa_shared_mlp with pool_k = n). */
PSA_API size_t psa_sa_group_all_workspace_bytes(int b, int n, int c, const psa_mlp* mlp);
PSA_API int psa_sa_group_all_infer(int b, int n, int c, const float* xyz, const float* points, const psa_mlp* mlp,
                                   float* out, void* workspace, size_t workspace_bytes, psa_stream_t stream);

/* Arithmetic of the grouped MLP.  Whenever the shapes allow -- set-abstraction levels with widths 64/128 (last width 64 or a
 * multiple of 128) and nsample 32/64/128 on tc_sa_dual_kernel, dense layers with N = 64 or a multiple of 128 on tc_dense2 /
 * tc_dense3 -- the layers after the first run on the tcgen05 tensor cores with fp32 accumulation in tensor memory; other shapes
 * run on the fp32-FMA kernels.  The fp32 operands are split into exactly representable 16-bit pieces:
 *   0 (default): two fp16 pieces per operand (22 mantissa bits), three MMAs per product  a1w2 + a2w1 + a1w1  -- the same error
 *      against fp64 as an fp32 FMA chain (1e-5 contract of the tests).  fp16 covers |v| < 65504: every kernel tracks the pieces
 *      it stores (weights too) and raises a device-side flag when a value leaves that range; the call then reruns the op with
 *      bf16x3 operands (launched unconditionally, a no-op unless the flag is set), so results are valid for any fp32 input.
 *   2: three bf16 pieces per operand, six MMAs per product (small terms first) -- any magnitude, twice the tensor work.
 *   1: fp32-FMA kernels only.
 * Weight images (psa_prepare_weight_image) are format-specific: psa_mlp_image_plan returns the format of the current mode in its
 * nt values; images of the other format are ignored (rebuilt per call).  The switch is process-global (two atomics: changing it while
 * other threads launch is race-free, but a call in flight may see either mode for its later layers): set it before launching
 * work, not concurrently with it. */
PSA_API int psa_set_mlp_mode(int mode);
PSA_API int psa_get_mlp_mode(void);

/* Training-mode front of a set-abstraction level ("variant F1"): ball query + group + centre + first 1x1 conv + bias in
 * one launch, writing the PRE-batch-norm activations (which training-mode BN needs in HBM once: batch statistics come
 * before the ReLU, pointnet2/utils/tf_util.py:512-531 with is_training=True) and, optionally, their per-channel sum and
 * sum of squares.  xyz (b,n,3), new_xyz (b,m,3), points (b,n,c) or NULL, w1 (3+c, C1) (xyz rows first), bias (C1) or
 * NULL -> pre (b,m,nsample,C1), idx (b,m,nsample), pts_cnt (b,m) or NULL, stats (2,C1) or NULL.  C1 in {64,128}.
 * Replaces query_ball_point + group_point x2 + tile/sub + concat + conv2d/bias_add (pointnet_util.py:44-50,117-123). */
PSA_API size_t psa_sa_conv1_prebn_workspace_bytes(int b, int n, int m, int c, int C1, int want_stats);
PSA_API int psa_sa_conv1_prebn(int b, int n, int m, int c, float radius, int nsample, const float* xyz,
                               const float* new_xyz, const float* points, const float* w1, const float* bias, int C1,
                               float* pre, int* idx, int* pts_cnt, float* stats, void* workspace,
                               size_t workspace_bytes, psa_stream_t stream);

/* Fused EdgeConv, inference mode (dgcnn/models/dgcnn.py:31-47 pattern): x (b,n,c), nn_idx (b,n,k) ->
 * out (b,n,C_L) = max_j MLP([x_i, x_j - x_i]); mlp->channels[0] must equal 2c.  A single-layer MLP is evaluated as
 * (W_a - W_b).x_i + W_b.x_j: one GEMM over the b*n POINTS plus a gather-max pass (k-fold fewer FLOPs than a conv over the
 * b*n*k edges); deeper MLPs use the fused gather + MLP + max kernel.  workspace: psa_edgeconv_workspace_bytes(). */
PSA_API size_t psa_edgeconv_workspace_bytes(int b, int n, int c, int k, const psa_mlp* mlp);
PSA_API int psa_edgeconv_infer(int b, int n, int c, int k, const float* x, const int* nn_idx, const psa_mlp* mlp,
                               float* out, void* workspace, size_t workspace_bytes, psa_stream_t stream);


/* DGCNN kNN graph with the X.X^T contraction on the tensor cores and an exact refine (csrc/knn_tc.cu): same result as
 * psa_knn_graph -- indices bit-identical to the canonical fp32 evaluation (dot as an fma chain over the channels,
 * adj = (|p|^2 + (-2 dot)) + |q|^2, k smallest, lower index first on ties; dgcnn/utils/tf_util.py:638-671) -- for
 * 128 <= n <= 2048, c <= 64, k <= 64; other shapes (or a workspace smaller than psa_knn_graph_workspace_bytes) run the
 * fp32 kernel of psa_knn_graph.  workspace: bf16x3 images of the clouds, their canonical norms, the exhaustive-row worklist. */
PSA_API size_t psa_knn_graph_workspace_bytes(int b, int n, int c, int k);
PSA_API int psa_knn_graph_ws(int b, int n, int c, int k, const float* x, int* nn_idx, void* workspace, size_t workspace_bytes,
                             psa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Training mode (SURVEY 8f rank 1): batch-statistics batch norm through every layer of a level and the
 * backward pass.  Reference semantics: pointnet2/utils/tf_util.py:155-185 (conv2d = matmul + bias, then
 * batch norm, then relu), :512-531 (tf.contrib.layers.batch_norm, is_training=True: batch mean, BIASED batch
 * variance, eps = 1e-3, moving averages updated in place with `decay`), pointnet_util.py:113-127 (MLP +
 * reduce_max), gradients tf_grouping.py:43-47 (GroupPointGrad = scatter-add by idx; index ops carry no
 * gradient, tf_sampling.py:23,58, tf_grouping.py:22,33), optimiser pointnet2/train.py:139-146 (Adam).
 * A level keeps ONE tensor per layer, the PRE-batch-norm activations y_l; everything else is recomputed
 * inside the GEMM operand loads (csrc/train_gemm.cuh).  All reductions (statistics, bias/BN gradients, weight
 * gradients, the GroupPointGrad scatter) are evaluated in a fixed order: results are bit-reproducible run to
 * run, unlike the reference's float atomicAdd scatters.
 * ------------------------------------------------------------------------------------------- */

/* Forward input of a layer: h[r][c] = relu(x[r][c] * scale[c] + shift[c]) * mask[r][c].
 * scale == NULL: identity (raw input, no relu).  mask == NULL: no dropout. */
typedef struct psa_act_in {
    const float* x;      /* (rows, ld) */
    long long ld;
    const float* scale;  /* (C) batch-norm scale = gamma / sqrt(var + eps) of the layer that produced x, or NULL */
    const float* shift;  /* (C) beta - mean * scale */
    const float* mask;   /* (rows, ld) dropout mask holding 0 or 1/keep_prob, or NULL */
    int relu;
} psa_act_in;

/* Gradient w.r.t. a layer's PRE-batch-norm output: dy[r][c] = ca[c] * dz[r][c] + cb[c] * y[r][c] + cc[c]
 * (the batch-norm backward with the batch sums folded into three per-channel constants, see
 * psa_bn_bwd_coeffs), dz = gradient w.r.t. the batch-norm output after the relu mask [y*s+t > 0]:
 *   mode 0: dz = dh[r][c] (* mask[r][c])                      dense incoming gradient
 *   mode 1: dz = dp[g][c] if argk[g][c] == r - g*pool_k and pv[g][c] > 0 else 0,  g = r / pool_k
 *           (max-pool routing: dp = gradient of the pooled output, pv = pooled value, argk = winning row).
 * ca == NULL: dy = dz (layer without batch norm).  s == NULL: no relu mask. */
typedef struct psa_grad_in {
    const float* y;      /* (rows, ld) pre-BN activations of this layer */
    long long ld;
    const float* s;      /* (C) BN scale / shift of this layer, or NULL */
    const float* t;
    int relu;
    const float* ca;     /* (C) or NULL */
    const float* cb;
    const float* cc;
    const float* dh;     /* mode 0: (rows, ld_dh) */
    long long ld_dh;
    const float* mask;   /* mode 0: dropout mask on dh, or NULL */
    const float* dp;     /* mode 1: (rows / pool_k, C) */
    const float* pv;
    const int* argk;
    int pool_k;
    int C;
    int mode;
} psa_grad_in;

/* y (rows, N) = in (rows, K) . W (K, N) + bias; stats (2, N) = per-channel [sum, sum of squares] of y (or NULL).
 * workspace: psa_train_dense_workspace_bytes(rows, K, N). */
PSA_API size_t psa_train_dense_workspace_bytes(long long rows, int K, int N);
PSA_API int psa_train_dense_fwd(long long rows, int K, int N, const psa_act_in* in, const float* W, const float* bias,
                                float* y, float* stats, void* workspace, size_t workspace_bytes, psa_stream_t stream);
/* dx (rows, K - col_skip) = dy (rows, N) . W^T restricted to input channels >= col_skip (the xyz channels of a
 * concatenated input carry no gradient that anyone consumes). */
PSA_API int psa_train_dense_bwd_input(long long rows, int K, int N, const psa_grad_in* g, const float* W, float* dx,
                                      long long ld_dx, int col_skip, void* workspace, size_t workspace_bytes,
                                      psa_stream_t stream);
/* dW (K, N) = in^T . dy, contraction over the rows in fixed split order (deterministic). */
PSA_API int psa_train_dense_bwd_weight(long long rows, int K, int N, const psa_act_in* in, const psa_grad_in* g,
                                       float* dW, void* workspace, size_t workspace_bytes, psa_stream_t stream);

/* Pooling of (groups*pool_k, C) rows over each run of pool_k rows, the modes of pointnet_sa_module other than the fused max
 * (pointnet2/utils/pointnet_util.py:126-146): mode 0 max, 1 avg (reduce_mean), 2 weighted_avg with weights
 * exp(-5 d) / sum exp(-5 d), d = dist (groups*pool_k) = the norm of each row's centred coordinates.  out (groups, C). */
PSA_API int psa_pool_rows(long long groups, int pool_k, int C, int mode, const float* x, const float* dist, float* out,
                          psa_stream_t stream);

/* Bias gradient of a layer that is NOT followed by batch norm: db (N) = sum_r dy[r][:].  (Under batch norm the conv / fc bias
 * has an identically zero gradient -- sum_r dy = 0 -- and the training path writes exact zeros there.) */
PSA_API int psa_train_bias_grad(long long rows, int N, const psa_grad_in* g, float* db, psa_stream_t stream);

/* Batch statistics -> BN affine.  stats (2, C) sums over `count` rows; gamma, beta (C) ->
 * scale = gamma / sqrt(var + 1e-3), shift = beta - mean * scale, mean_inv (2, C) = [mean, 1/sqrt(var + eps)];
 * moving_mean / moving_var (C, may be NULL) <- decay * moving + (1 - decay) * batch  (tf_util.py:526-531). */
PSA_API int psa_bn_finalize(int C, long long count, const float* stats, const float* gamma, const float* beta,
                            float decay, float* moving_mean, float* moving_var, float* scale, float* shift,
                            float* mean_inv, psa_stream_t stream);

/* relu(BN(y)) then max over each run of pool_k rows: pooled (groups, C), argk (groups, C) = first winning row. */
PSA_API int psa_train_pool_fwd(long long groups, int pool_k, int C, const float* y, const float* scale,
                               const float* shift, float* pooled, int* argk, psa_stream_t stream);

/* Batch-norm backward sums of a layer: dbeta[c] = sum_r dz, dgamma[c] = sum_r dz * xhat (g->ca/cb/cc are ignored),
 * and the coefficients ca = gamma*inv, cb = -gamma*inv^2*dgamma/rows, cc = gamma*inv*(mean*inv*dgamma - dbeta)/rows
 * that make psa_grad_in evaluate dy.  workspace: psa_bn_bwd_workspace_bytes(C). */
PSA_API size_t psa_bn_bwd_workspace_bytes(int C);
PSA_API int psa_bn_bwd_coeffs(long long rows, int C, const psa_grad_in* g, const float* gamma, const float* mean_inv,
                              float* dgamma, float* dbeta, float* ca, float* cb, float* cc, void* workspace,
                              size_t workspace_bytes, psa_stream_t stream);

/* Backward of the fused first layer of a set-abstraction level (psa_sa_conv1_prebn): with dy0 = g over the
 * b*m*nsample grouped rows,  dW_xyz (3, C1) = sum_r (xyz[idx_r] - new_xyz[q_r])^T dy0[r]  and, if dU != NULL,
 * dU (b*n, C1) = GroupPointGrad(dy0, idx) (tf_grouping_g.cu:61-78) as a stable counting sort of the (row -> point)
 * entries followed by an ordered gather (each source point adds its rows in ascending row order: deterministic).  The feature part of the layer then is two dense products on the b*n
 * POINTS: dpoints = dU . W1[3:]^T and dW1[3:] = points^T . dU.  workspace: psa_sa_conv1_bwd_workspace_bytes(...). */
PSA_API size_t psa_sa_conv1_bwd_workspace_bytes(int b, int n, int m, int nsample, int C1, int want_dU);
PSA_API int psa_sa_conv1_bwd(int b, int n, int m, int nsample, int C1, const float* xyz, const float* new_xyz,
                             const int* idx, const psa_grad_in* g, float* dW_xyz, float* dU, void* workspace,
                             size_t workspace_bytes, psa_stream_t stream);

/* Training-mode front of a feature-propagation module (pointnet2/utils/pointnet_util.py:199-229 with three_nn / three_interpolate,
 * 3d_interpolation/tf_interpolate.cpp:60-127, inside pointnet2/models/pointnet2_cls_bga.py:51-53).  The first 1x1 conv of the module
 * distributes over the (linear) interpolation:
 *   y = [interp, skip] . W1 + b = sum_i w_i U[idx_i] + skip . W1[C_a:] + b,   U = P2 . W1[:C_a]  (one row per KNOWN point)
 * so the (b, n, C_a) interpolated tensor and the concatenation never exist.  U (b, m, C1) comes from psa_train_dense_fwd (its
 * psa_act_in applies the producer's batch norm + relu on load), as does the skip product.  This call does, in one pass:
 * three_nn of xyz1 (b,n,3) unknown against xyz2 (b,m,3) known + the inverse-distance weights (arithmetic and results bit-identical to
 * psa_three_nn_interpolate), pre (b,n,C1) = [pre if accumulate, else bias (or 0 for NULL)] + (U[i1] w1 + U[i2] w2) + U[i3] w3,
 * idx / weight (b,n,3) for the backward, and, if stats != NULL, stats (2, C1) = per-channel [sum, sum of squares] of pre (fixed-order
 * CTA partials added in fp64).  Slots beyond m (m < 3) have weight 0 and idx 0.  C1 a multiple of 4, at most 512; m >= 1.
 * workspace: psa_fp_conv1_prebn_workspace_bytes(b, n, C1) when stats != NULL. */
PSA_API size_t psa_fp_conv1_prebn_workspace_bytes(int b, int n, int C1);
PSA_API int psa_fp_conv1_prebn(int b, int n, int m, int C1, const float* xyz1, const float* xyz2, const float* U, const float* bias,
                               int accumulate, float* pre, int* idx, float* weight, float* stats, void* workspace,
                               size_t workspace_bytes, psa_stream_t stream);

/* Backward of psa_fp_conv1_prebn: dU (b, m, C1) = ThreeInterpolateGrad(dy0, idx, weight) (tf_interpolate.cpp:131-153), dy0 = g over the
 * b*n unknown rows (mode 0, evaluated on load: the batch-norm backward coefficients are applied there).  Ordered like
 * psa_three_interpolate_grad (stable counting sort by destination, each known point adds round(dy0 * w) of its entries 3*row + slot
 * in ascending order): with a plain g (dy0 = dh) the result is bit-identical to psa_three_interpolate_grad(dh).  The rest of the
 * layer's backward is dense: dW1[:C_a] = P2^T . dU and dP2 = dU . W1[:C_a]^T over the b*m known points, dW1[C_a:] = skip^T . dy0 and
 * dskip = psa_train_dense_bwd_input(..., col_skip = C_a).  workspace: psa_fp_conv1_bwd_workspace_bytes(b, n, m). */
PSA_API size_t psa_fp_conv1_bwd_workspace_bytes(int b, int n, int m);
PSA_API int psa_fp_conv1_bwd(int b, int n, int m, int C1, const int* idx, const float* weight, const psa_grad_in* g, float* dU,
                             void* workspace, size_t workspace_bytes, psa_stream_t stream);

/* Joint loss of pointnet2_cls_bga.get_loss (pointnet2/models/pointnet2_cls_bga.py:78-93): class logits (b, c) with labels (b) int32,
 * per-point seg logits (b, n, 2) with a binary mask (b, n) int32 ->
 *   loss (3) = [(1-w) classify + w seg, classify = mean_b CE, seg = mean over b*n points of the 2-way CE],
 *   dcls (b, c) = (1-w) (softmax - onehot) / b,  dseg (b, n, 2) = w (softmax - onehot) / (b n).
 * Sums in a fixed order (per-block trees, blocks added in order, fp64).  A label or mask value outside its range gives NaN.
 * workspace: psa_cls_seg_xent_workspace_bytes(b, n). */
PSA_API size_t psa_cls_seg_xent_workspace_bytes(int b, int n);
PSA_API int psa_cls_seg_xent(int b, int c, int n, const float* cls_logits, const int* labels, const float* seg_logits, const int* mask,
                             float seg_weight, float* loss, float* dcls, float* dseg, void* workspace, size_t workspace_bytes,
                             psa_stream_t stream);

/* Mean sparse softmax cross-entropy (pointnet2_cls_ssg.py:50-57) and its gradient: logits (b, c), labels (b) int32 ->
 * loss (1), dlogits (b, c) = (softmax - onehot) / b. */
PSA_API int psa_softmax_xent(int b, int c, const float* logits, const int* labels, float* loss, float* dlogits,
                             psa_stream_t stream);

/* tf.train.AdamOptimizer step over one flat parameter vector (pointnet2/train.py:139-146):
 * g = grad * grad_scale; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr sqrt(1-b2^t)/(1-b1^t) m / (sqrt(v) + eps). */
PSA_API int psa_adam_step(long long count, float* params, const float* grads, float* m, float* v, float lr, float beta1,
                          float beta2, float eps, int step, float grad_scale, psa_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PSA_H_ */
