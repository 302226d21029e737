/* pcreid.h -- C ABI of libpcreid_sm100.so, the B200 (sm_100a) replacement for the data-parallel hot
 * path of bentherien/point-cloud-reid.  Plain pointers and sizes only; every pointer is a DEVICE
 * pointer unless stated; `stream` is a cudaStream_t passed as void*.  Every function is asynchronous
 * on `stream`, allocates nothing, keeps no global state and returns PCREID_OK (0) or an error code
 * (the reference launchers fprintf + exit(-1) instead, e.g. knn_cuda.cu:110-114).
 *
 * Citations are into the reference tree (mmdet3d/...).  Section A is the op-level boundary: each entry
 * point takes exactly the arguments of the reference's `*_kernel_launcher` it replaces, so the
 * reference's pybind wrapper (ops/<op>/src/<op>.cpp) can call it unchanged (INTEGRATION.md).
 * Section B is the model-level boundary: the kernels the Python modules in
 * point-cloud-reid_b200/models call from ReIDNet.forward / backbone.forward / match_forward_inference.
 */
#ifndef PCREID_H_
#define PCREID_H_

#ifdef __cplusplus
extern "C" {
#endif

#define PCREID_OK 0
#define PCREID_ERR_ARG 1          /* null pointer / bad size */
#define PCREID_ERR_LAUNCH 2       /* cudaGetLastError() != cudaSuccess after the launch */
#define PCREID_ERR_UNSUPPORTED 3  /* shape outside what the kernels were built for */

int pcreid_abi_version(void);

/* ------------------------------------------------------------------ A. mmdet3d point ops ------- */

/* replaces furthest_point_sampling_kernel_launcher(b,n,m,dataset,temp,idxs,stream)
 * (ops/furthest_point_sample/src/furthest_point_sample_cuda.cu:143-211; python
 * furthest_point_sample.py:7-44).  xyz (b,n,3) f32, temp (b,n) f32 scratch pre-filled with 1e10 by
 * the caller (may be NULL: treated as 1e10), idx (b,m) i32.  First index is 0; ties follow the
 * reference's shared-memory tree: min (bitreverse(k mod bs), k), bs = pcreid_fps_block_size(n). */
int pcreid_fps(int b, int n, int m, const float* xyz, float* temp, int* idx, void* stream);
/* replaces furthest_point_sampling_with_dist_kernel_launcher (same file :333-400): dist (b,n,n). */
int pcreid_fps_with_dist(int b, int n, int m, const float* dist, float* temp, int* idx, void* stream);
int pcreid_fps_block_size(int n); /* host helper: opt_n_threads(n), same file :11-15 */
/* replaces the torch-path farthest_point_sample (models/pointnet2_utils.py:116-137; a Python loop of npoint steps over
 * index / sub / pow / sum / masked assignment / max there), the SA sampling with sampling="FPS": idx[b,0] = start[b] (the
 * reference draws it with torch.randint on the host), distance (dx*dx + dy*dy) + dz*dz without contraction, running minimum
 * initialised to 1e10, arg-max with the lowest index among tied maxima (torch.max on the CPU).  idx (b,m) int32. */
int pcreid_fps_torch(int b, int n, int m, const float* xyz, const int* start, int* idx, void* stream);
/* replaces calc_square_dist (ops/furthest_point_sample/utils.py:4-31; torch sum / matmul / sqrt there): the (b,n,m) feature
 * distance matrix the F-FPS / FS samplers (points_sampler.py:124-157) pass to furthest_point_sample_with_dist.
 * a (b,n,c), b (b,m,c) point-major; out[b,i,j] = |a_i|^2 + |b_j|^2 - 2 a_i.b_j (fma chains over c ascending);
 * norm != 0: sqrt(.) / c. */
int pcreid_pairwise_sqdist(int b, int n, int m, int c, const float* a, const float* bm, float* out, int norm, void* stream);

/* replaces knn_kernel_launcher(b,n,m,nsample,xyz,new_xyz,idx,dist2,stream) (ops/knn/src/knn_cuda.cu:97-116;
 * python knn.py:7-71).  xyz (b,n,3), new_xyz (b,m,3), idx/dist2 (b,m,nsample); nsample <= 100.
 * Ascending distance; exact ties resolved exactly as the reference's max-heap does. */
int pcreid_knn(int b, int n, int m, int nsample, const float* xyz, const float* new_xyz, int* idx, float* dist2, void* stream);
/* same search, idx/dist2 written as (b,nsample,m): the layout knn.py:62 returns */
int pcreid_knn_t(int b, int n, int m, int nsample, const float* xyz, const float* new_xyz, int* idx, float* dist2, void* stream);

/* replaces ball_query_kernel_launcher(b,n,m,min_radius,max_radius,nsample,new_xyz,xyz,idx,stream)
 * (ops/ball_query/src/ball_query_cuda.cu:56-82; python ball_query.py:7-54).  idx (b,m,nsample) must be
 * zero-filled by the caller (ball_query.py:41); rows without a hit are left untouched. */
int pcreid_ball_query(int b, int n, int m, float min_radius, float max_radius, int nsample,
                      const float* new_xyz, const float* xyz, int* idx, void* stream);
/* replaces the torch-path query_ball_point (models/pointnet2_utils.py:218-240; arange / square_distance / sort / mask there),
 * the grouping of the ReID backbone's SA layers when use_knn=False: expansion-form distance of square_distance op for op,
 * a point is kept unless d2 > r2 (r2 = fp32(radius ** 2)), first nsample kept indices in ascending order, padded with the
 * first; idx (b,m,nsample) int32; a row without any kept point is filled with n (as the reference's sort leaves it). */
int pcreid_query_ball_point(int b, int n, int m, float r2, int nsample, const float* new_xyz, const float* xyz, int* idx,
                            void* stream);

/* replaces group_points_kernel_launcher(b,c,n,npoints,nsample,points,idx,out,stream)
 * (ops/group_points/src/group_points_cuda.cu:81-100): out[b,c,s,j] = points[b,c,idx[b,s,j]]. */
int pcreid_group_points(int b, int c, int n, int npoints, int nsample, const float* points, const int* idx, float* out, void* stream);

/* the body of QueryAndGroup.forward (ops/group_points/group_points.py:93-118) after the index query, in one pass over the
 * (b, c+3, npoints, nsample) result instead of the reference's grouping_operation x2 + transpose + sub + div + cat:
 *   out[b, 0:3, s, j]  = (xyz[b, idx[b,s,j], :] - center_xyz[b, s, :]) (/ divide_by when divide_by != 0: normalize_xyz)   if use_xyz
 *   out[b, 3*use_xyz + ch, s, j] = features[b, ch, idx[b,s,j]]                                   if features != NULL (b,c,n)
 *   grouped_xyz[b, 0:3, s, j] = xyz[b, idx[b,s,j], :]                                             if grouped_xyz != NULL
 * xyz (b,n,3), center_xyz (b,npoints,3), idx int32 (b,npoints,nsample).  Bit-identical to the reference's op chain. */
int pcreid_query_group(int b, int c, int n, int npoints, int nsample, const float* xyz, const float* center_xyz, const float* features,
                       const int* idx, int use_xyz, float divide_by, float* out, float* grouped_xyz, void* stream);
/* replaces gather_points_kernel_launcher(b,c,n,npoints,points,idx,out,stream)
 * (ops/gather_points/src/gather_points_cuda.cu:28-49): out[b,c,m] = points[b,c,idx[b,m]]. */
int pcreid_gather_points(int b, int c, int n, int npoints, const float* points, const int* idx, float* out, void* stream);
/* Crop -> centre -> resample front-end (csrc/frontend.cu; reference: models/trackers/deprecated/pc_utils.py:31-96 +
 * DepthInstance3DBoxes.points_in_boxes, core/bbox/structures/depth_box3d.py:256-282 +
 * ops/roiaware_pool3d/src/points_in_boxes_cuda.cu:24-105).  pts (P, >=3) with row stride pts_stride floats, boxes (B, 7)
 * = (x, y, z centre, dx, dy, dz, yaw) in the depth frame.
 *   pcreid_crop_mask:   mask (B, ntiles, 32) uint32, bit i of word w <-> point tile*1024 + 32 w + i lies in box b;
 *                       counts (B, ntiles) int32; ntiles = pcreid_crop_tiles(P).
 *   pcreid_crop_gather: prefix (B, ntiles+1) = exclusive scan of counts; rank (B, N) int64 in [0, length_b): out (B, N, 3)
 *                       = box-frame coordinates of the rank-th in-box point (point order), zeros where length_b == 0. */
int pcreid_crop_tiles(int P);
int pcreid_crop_mask(int P, int B, const float* pts, int pts_stride, const float* boxes, void* mask, int* counts, void* stream);
int pcreid_crop_gather(int P, int B, int N, const float* pts, int pts_stride, const float* boxes, const void* mask,
                       const int* prefix, const long long* rank, float* out, void* stream);

/* replaces three_nn_kernel_launcher(b,n,m,unknown,known,dist2,idx,stream) (ops/interpolate/src/three_nn_cuda.cu:68-90):
 * the three nearest known (B,M,3) points of every unknown (B,N,3) point, ascending (d2, index); dist2 (B,N,3) SQUARED
 * distances (the Python wrapper takes the root, three_nn.py:37), idx int32 (B,N,3); unfilled slots (M < 3) = (0, +inf). */
int pcreid_three_nn(int b, int n, int m, const float* unknown, const float* known, float* dist2, int* idx, void* stream);
/* replaces three_interpolate_kernel_launcher(b,c,m,n,points,idx,weight,out,stream)
 * (ops/interpolate/src/three_interpolate_cuda.cu:40-62): out[b,c,n] = sum_j weight[b,n,j] * points[b,c,idx[b,n,j]]. */
int pcreid_three_interpolate(int b, int c, int m, int n, const float* points, const int* idx, const float* weight, float* out,
                             void* stream);

/* ------------------------------------------------------------------ B. encoder / match path ---- */
/* All feature tensors are channel-major per object, exactly the reference's (B, C, N) layout:
 * element (b, c, n) at  base + map(b)*bs + c*ld + n.  `map` (optional) is an int32 object-gather map,
 * used to score pairs without materialising `feat[pairs[:,0]]` (tracking_point_reid.py:110).        */

/* torch-path kNN of the ReID backbones (models/pointnet2_utils.py:169-216 square_distance + argsort):
 * expansion-form distance, canonical ascending (d, idx) order.  idx (b,m,k) i32. */
int pcreid_knn_point(int b, int n, int m, int k, const float* xyz, const float* new_xyz, int* idx, void* stream);
/* The same neighbours as pcreid_knn_point as an UNORDERED set (the order inside idx[b, q, :] is unspecified): the k
 * nearest points with the ordered kernel's tie rule at the k-th boundary (equal distances: lower index first).  For
 * consumers that max-pool over the neighbours (PointNetSetAbstractionEdgeSA, pointnet2_utils.py:333-357).
 * k <= n <= 1024, else PCREID_ERR_UNSUPPORTED. */
int pcreid_knn_point_set(int b, int n, int m, int k, const float* xyz, const float* new_xyz, int* idx, void* stream);
/* DGCNN kNN (models/dgcnn_orig.py:22-28): x (b,c,n) channel-major with object stride x_bs, k largest of
 * pd = -|xi|^2 + 2 xi.xj - |xj|^2, lower index first on ties.  idx (b,n,k) i32. */
int pcreid_knn_feature(int b, int c, int n, int k, const float* x, long long x_bs, int* idx, void* stream);

enum { PCREID_ACT_NONE = 0, PCREID_ACT_RELU = 1, PCREID_ACT_LEAKY02 = 2, PCREID_ACT_ELU1 = 3 };

/* Y[b,co,n] = act( sum_k W1[k,co] X1[b,k,n] + sum_k W2[k,co] X2[b,k,n] + bias[co] (+R) ) (+R)
 * = every nn.Linear / 1x1 Conv1d / Conv2d(+folded eval BatchNorm) on the path.  Weights are k-major
 * [K, CO] (the transpose of torch's [CO, K]); per-object weights via w*_bs / w1_map. */
typedef struct pcreid_linear_args {
  int B, rows, CO, K1, K2;
  const float* X1; long long x1_bs; int ldx1; int x1_pm; const int* x1_map;   /* x*_pm=1: point-major (rows,K) */
  const float* X2; long long x2_bs; int ldx2; int x2_pm; const int* x2_map;
  const float* W1; long long w1_bs; const int* w1_map;
  const float* W2; long long w2_bs;
  const float* bias;
  const float* R; long long r_bs; int ldr; const int* r_map; int res_after_act;
  int act;
  float* Y; long long y_bs; int ldy; int y_pm;   /* y_pm=1: Y written point-major (rows, CO), ldy = row stride */
} pcreid_linear_args;
int pcreid_cn_linear(const pcreid_linear_args* args, void* stream);
/* same contract on the tensor cores (tcgen05 kind::tf32, fp32 accumulate): fast mode.  Returns PCREID_ERR_UNSUPPORTED
 * for shapes it was not built for (object maps, point-major inputs, K < 8);
 * callers then use pcreid_cn_linear. */
int pcreid_cn_linear_tc(const pcreid_linear_args* args, void* stream);

/* GroupNorm over channel groups per (object, point) -- LayerNorm is G=1 (eps 1e-5, torch default):
 * Y = act( GN(X)*gamma + beta (+R) ).  Used for nn.LayerNorm (pointnet2_utils.py:87-88, attention.py:187-188)
 * and LinearRes' GroupNorm (lanegcn_nets.py:206-221). */
typedef struct pcreid_norm_args {
  int B, rows, C, G;
  const float* X; long long x_bs; int ldx;
  const float* gamma; const float* beta;
  const float* R; long long r_bs; int ldr; const int* r_map;
  int act;
  float* Y; long long y_bs; int ldy;
} pcreid_norm_args;
int pcreid_cn_groupnorm(const pcreid_norm_args* args, void* stream);

/* Tail of the match head in one pass over the pairs (the second GroupNorm + identity shortcut + ReLU of LinearRes followed by
 * the final Linear(C, 1): mmdet3d/models/lanegcn_nets.py:228-241 `LinearRes.forward`, head configs
 * configs_reid/.../reid_pts_point-transformer_point-cat.py:24-25):
 *   y[:, p] = relu(GroupNorm_G(X[:, p]) * gamma + beta + R[:, p]),   out[p] = w . y[:, p] + bias
 * X, R: (C, rows) channel-major with channel strides ldx / ldr; the same GroupNorm arithmetic as pcreid_cn_groupnorm (eps 1e-5,
 * biased variance).  y is never written. */
int pcreid_gn_res_relu_dot(int rows, int C, int G, const float* X, int ldx, const float* gamma, const float* beta,
                           const float* R, int ldr, const float* w, float bias, float* out, void* stream);

/* Second generation of pcreid_cn_linear_tc (csrc/cn_linear_tc2.cu): warp-specialised persistent tf32 GEMM (activation
 * loader warps, bulk-TMA weight loader, MMA issuer, epilogue warps over a double-buffered TMEM accumulator).  Same
 * contract; the weights are ALSO passed as operand images W*img[(k/4)][co][k%4] (fp32, K a multiple of 8).  Shared
 * (not per-object) weights, channel-major inputs, no object maps; else PCREID_ERR_UNSUPPORTED. */
int pcreid_cn_linear_tc2(const pcreid_linear_args* args, const float* W1img, const float* W2img, int n_sms, void* stream);

/* Third generation (csrc/cn_linear_tma.cu): the same contract with both operands staged by TMA tensor maps
 * (cp.async.bulk.tensor, 128-byte swizzle) directly from the channel-major activations and the k-major weights as
 * MN-major tcgen05 kind::tf32 operands -- no weight images, any K (zero-filled by the TMA unit), shared or per-object
 * weights, object maps (x1_map / x2_map / w1_map / r_map) as the third box coordinate.  x*_objs / w1_objs: number of objects in
 * the mapped source tensors (the bound of the tensor map's third extent; ignored without a map).
 * flags: PCREID_TMA_TF32_MAPS  activation maps typed TFLOAT32 (the TMA unit rounds fp32 -> tf32 instead of the tensor
 *                             core truncating), PCREID_TMA_ROUND_OUT  Y rounded to tf32 (feeds another tf32 GEMM).
 * PCREID_ERR_UNSUPPORTED: point-major inputs or outputs, CO < 32, CO % 4, rows % 4, row / object strides that are not multiples of 4 floats,
 * unaligned base pointers, no driver entry point for cuTensorMapEncodeTiled. */
#define PCREID_TMA_TF32_MAPS 1
#define PCREID_TMA_ROUND_OUT 2
#define PCREID_TMA_TILE128 4     /* A/B knob: never use the 256-channel tiles chosen for K >= 256 and CO >= 256 */
int pcreid_cn_linear_tma(const pcreid_linear_args* args, long long x1_objs, long long x2_objs, long long w1_objs, int flags, int n_sms,
                         void* stream);
/* fp32-grade variant of the same kernel ("3 x tf32"): every operand is split hi + lo (hi = the 19 bits the tensor core reads of the
 * raw fp32 word, lo = the exact remainder), three MMAs per K step (lo.hi + hi.lo + hi.hi) into the fp32 accumulator.  W*lo: the
 * weights' lo parts (same shapes / strides as W1 / W2), `w - float(bits(w) & 0xffffe000)`; the activations' lo tiles are made in
 * shared memory.  Matches pcreid_cn_linear to ~1e-6 relative.  Same shape restrictions as pcreid_cn_linear_tma. */
int pcreid_cn_linear_tma_x3(const pcreid_linear_args* args, const float* W1lo, const float* W2lo, long long x1_objs, long long x2_objs,
                            long long w1_objs, int n_sms, void* stream);

/* LinearAttention (pointnet2_utils.py:14-47, attention.py:19-54), split in two kernels:
 * kv:    Wkv[b] (d x d, k-major, block diagonal per head) = sum_s (elu(k_s)+1) (x) (v_s / S);  ksum[b] (d)
 * scale: Qs[b,c,n] = (elu(q)+1) * S / ( (elu(q_h)+1) . ksum_h + 1e-6 )
 * so that message = cn_linear(X1=Qs, W1=Wkv (per object)). */
int pcreid_linattn_kv(int B, int S, int d, int H, const float* K, long long k_bs, int ldk,
                      const float* V, long long v_bs, int ldv, float* Wkv, float* ksum, void* stream);
int pcreid_linattn_scale(int B, int rows, int d, int H, int S, const float* Q, long long q_bs, int ldq, const int* q_map,
                         const float* ksum, const int* ksum_map, float* Qs, long long qs_bs, int ldqs, void* stream);

/* local_self_attention core (attention.py:221-296, the 'xcorr' match type): every point attends its knum feature-space
 * neighbours (idx from pcreid_knn_feature) with one query: out[b,n,h,:] = sum_j w_j v_j / (sum_j w_j + 1e-6),
 * w_j = (elu(q_h)+1).(elu(k_jh)+1).  qkv point-major (B, N, 3C) rows [q | k | v] pre-activation, out point-major (B, N, C).
 * C a multiple of 32 up to 128, H in {1, 2, 4}. */
int pcreid_local_linattn(int B, int N, int C, int H, int knum, const float* qkv, const int* idx, float* out, void* stream);

/* pooling over points (ReIDNet.get_pooled_feats, ReIDNet.py:526-534; PointNet max-pool pointnet.py:31,70).
 * mode 0: out[b, c] = max_n, out[b, C + c] = mean_n over the rows of X1 (and X2 if given: 'point-cat');
 * mode 1: max only.  Output element (b, c) at out + b*ob + c*oc. */
int pcreid_cn_pool(int B, int C, int rows1, const float* X1, long long x1_bs, int ldx1,
                   int rows2, const float* X2, long long x2_bs, int ldx2,
                   int mode, float* out, long long ob, long long oc, void* stream);
/* 'max' pool_type of the reference: MaxPool1d over the CHANNEL axis (ReIDNet.py:527-528, 455-456):
 * out[b, n] = max_c X[b, c, n]; element (b, n) at out + b*ob + n*on. */
int pcreid_cn_chanmax(int B, int C, int rows, const float* X, long long x_bs, int ldx, float* out, long long ob, long long on, void* stream);

/* Fused set-abstraction edge MLP (PointNetSetAbstractionEdgeSA.forward, pointnet2_utils.py:333-357) after the
 * first 1x1 conv has been factorised into a per-point term P1 and a per-centre term Cc:
 *   out[b,c,s] = max_j relu(W3 relu(W2 relu(P1[b,:,idx[b,s,j]] + Cc[b,:,s]) + b2) + b3)[c]
 * P1 (b,C,n), Cc (b,C,S), idx (b,S,k) i32, W2/W3 k-major (C,C) with eval BatchNorm folded, out (b,C,S). */
int pcreid_sa_edge_mlp(int B, int C, int N, int S, int k, const float* P1, const float* Cc, const int* idx,
                       const float* W2, const float* b2, const float* W3, const float* b3, float* out, void* stream);

/* Unfused SA edge path for channel counts above the fused kernel's tile (C > 128: the mul=2 / mul=4 variants,
 * configs_reid/_base_/reidentifiers/reid_pts_point-transformer-{1.5M,7M}_point-cat.py):
 *   edge_build: H1[b,c,s*k+j] = relu(P1[b,c,idx[b,s,j]] + Cc[b,c,s])  (P1 (B,C,N), Cc (B,C,S), idx int32 (B,S,k), H1 (B,C,S*k));
 *   seg_max:    out[i] = max_j x[i*k + j]  (rows = B*C*S).  pointnet2_utils.py:353-357. */
int pcreid_edge_build(int B, int C, int N, int S, int k, const float* P1, const float* Cc, const int* idx, float* out, void* stream);
int pcreid_seg_max(long long rows, int k, const float* x, float* out, void* stream);
/* pool_mod='avg' of the mmdet3d SA modules (ops/pointnet_modules/point_sa_module.py:158-160, F.avg_pool2d over the k
 * samples): out[i] = (sum_j x[i*k + j]) / k, summed in sample order. */
int pcreid_seg_mean(long long rows, int k, const float* x, float* out, void* stream);

/* EdgeConv gather-max (dgcnn_orig.py:31-54,129-147 with the bias-free conv factorised):
 *   out[b,c,i] = act( max_j P[b,c,idx[b,i,j]] + Q[b,c,i] ),  element (b,c,i) at out + b*o_bs + c*ldo + i */
int pcreid_edge_gather_max(int B, int C, int N, int k, const float* P, const float* Q, const int* idx, int act,
                           float* out, long long o_bs, int ldo, void* stream);

/* Fused 'concat' match head over ALL pairs (ReIDNet.py:415-419,455-458 + LinearRes/Linear,
 * lanegcn_nets.py:228-241) without materialising the T x D x 2E pair tensor:
 *   logit[t,d] = w . relu( GN2(W2 relu(GN1(A[t] + Bv[d]))) + [e_t ; e_d] ) + b0
 * A (T,Hd) = W1[:, :E] e_t, Bv (D,Hd) = W1[:, E:] e_d (row-major, from cn_linear), E_t (T,E), E_d (D,E),
 * Hd = 2E <= 256, G groups.  mask (T,D) u8 optional: 0 -> logit 0 (class gating,
 * tracking_point_reid.py:15-33).  out (T,D) f32 row-major. */
/* tensor-core ("fast") version for the shipped head LinearRes(256, 256, GN 32 groups) + Linear(256, 1), E = 128:
 * W2img = bf16 K-major operand image [k/8][256 n][8] of linear2.weight (csrc/concat_tc.cu); other arguments as below. */
int pcreid_pair_concat_head_tc(int T, int D, int E, int G, const float* A, const float* Bv, const float* Et, const float* Ed,
                               const void* W2img, const float* g1, const float* be1, const float* g2, const float* be2,
                               const float* w, float b0, const unsigned char* mask, float* out, int n_ctas, void* stream);
int pcreid_pair_concat_head(int T, int D, int E, int G, const float* A, const float* Bv, const float* Et, const float* Ed,
                            const float* W2, const float* g1, const float* be1, const float* g2, const float* be2,
                            const float* w, float b0, const unsigned char* mask, float* out, void* stream);

/* Gated linear assignment of tracks to detections (csrc/assign.cu), the association step after the (T, D) logits: B problems
 * of score (B, T, D) f32 (higher = more alike), mask (B, T, D) u8 or NULL (all admissible), threshold min_score.  A pair is
 * admissible when mask != 0, the score is finite and score > min_score; its weight is double(score) - double(min_score).
 * Each problem gets a matching of admissible pairs of maximum total weight (each track and detection at most once):
 * det_for_track (B, T) / track_for_det (B, D) int32, -1 = unmatched.  Among several optimal matchings the choice is
 * deterministic and per problem (independent of the other problems of the call).  One CTA per problem: shortest augmenting
 * paths (Jonker-Volgenant / Crouse) with float64 duals.  work: B * pcreid_lsap_workspace_bytes(T, D) bytes of device scratch.
 * 0 <= T, D <= 4096 and B <= 65535, else PCREID_ERR_UNSUPPORTED; a non-finite min_score is PCREID_ERR_ARG. */
int pcreid_lsap_workspace_bytes(int T, int D);   /* per problem; -1 outside the supported shapes */
int pcreid_lsap(int B, int T, int D, const float* score, const unsigned char* mask, float min_score, int* det_for_track,
                int* track_for_det, void* work, void* stream);

/* ------------------------------------------------------------------ B'. fused tensor-core match path --- */
/* Tensor-core modes of the xcorr_eff head (csrc/pair_tc.cu, csrc/pair_tc2.cu): tcgen05 kind::f16 GEMMs with fp32
 * accumulation and fp32 norms.  `fmt` selects the 16-bit operand format of EVERY operand image of a call chain:
 *   PCREID_FMT_BF16  "fast" mode      (8-bit significand;  |dlogit| <= 3e-2)
 *   PCREID_FMT_F16   "parity_tc" mode (11-bit significand = tf32's; |dlogit| <= 5e-3; operands are O(1): key/value sums are
 *                    stored scaled by 1/points -- kv_scale / att_eps below -- and conversions saturate)
 * Operand "images" are [k/8][row][8] tiles of 128 points x 64 channels (16 KB); d_model = 64, 2 heads.  Reference
 * arithmetic: corss_attention.forward (mmdet3d/models/attention.py:192-219), ReIDNet.xcorr_eff (ReIDNet.py:231-247),
 * get_pooled_feats (ReIDNet.py:526-534).  Host side: point-cloud-reid_b200/models/fused_pairs.py.
 * The host folds LayerNorm1's affine into the following Linear, centres the merge / mlp[2] weights over their output
 * channels (LayerNorm inputs become zero-mean), pre-scales q_proj by 1/ln 2 (bf16: 1/bf16(ln 2)), adds LayerNorm2's beta
 * to the residual image (stage 1: pcreid_pack_image_bias) or after the pooling (stage 2: pcreid_pool_finish2).
 * Weight blob layouts: pair_tc.cu (P1B_*), pair_tc2.cu (Q1A_*, Q2_*). */
#define PCREID_FMT_BF16 0
#define PCREID_FMT_F16 1
/* (B, C, N) channel-major fp32 -> [B][N/128][C/8][128][8] 16-bit (act: PCREID_ACT_NONE or PCREID_ACT_ELU1) */
int pcreid_pack_image(int B, int C, int N, const float* src, long long s_bs, int lds, int act, int fmt, void* dst, void* stream);
int pcreid_pack_image_bias(int B, int C, int N, const float* src, long long s_bs, int lds, const float* bias, int fmt, void* dst,
                           void* stream);
/* M (B,64,64) = blockdiag(KV) Wm^T rows + ksum (B,64) -> attention operand images (B, 10240 bytes: one [10][32][8] 16-bit image per head) */
int pcreid_pack_b7(int B, const float* M, const float* ksum, int fmt, void* dst, void* stream);
/* pool_part (P,2,128) -> pooled^T (128,P): max | mean over the 2*npts points of the point-cat pair tensor (+ beta2) */
int pcreid_pool_finish2(int P, int npts, const float* part, const float* bias /* (64) or NULL */, float* out, void* stream);
/* npts = points per object (any value >= 1; objects are zero-padded to a multiple of 128 rows inside the operand images).
 * att_eps = LinearAttention.eps (1e-6, attention.py:21) times the scale the template's key/value sums carry
 * (MK1 of pcreid_pack_b7 for phase 1a; kv_scale of phase 1b for phase 2). */
/* phase 1a: per (pair, direction) unit and 128-point tile of the search object: QF1 = elu(Wq h)+1 image, H = h + beta2 image
 * (both per object), MK1 = the template's stage-1 attention operand; W = [W0b.diag(g1) | W0a | W0b.beta1 - W0a.beta2] (N=128,
 * K=144) | centred W2 | LN2 gamma.  The search object's own term W0a.h is part of the K = 144 GEMM (no precomputed U image). */
int pcreid_pair_p1a2(int n_units, int npts, int role, int fmt, float att_eps, const int* u_search, const int* u_templ,
                     const int* u_slot, const void* QF1, const void* H, const void* MK1, const void* W, void* A_out,
                     int n_ctas, void* stream);
int pcreid_pair_p1b_n(int n_units, int npts, int role, int fmt, float kv_scale, const int* u_search, const int* u_templ,
                      const int* u_slot, const void* PV, const void* W, void* A_out, void* B7_out, int n_ctas, void* stream);
int pcreid_pair_p2y(int n_units, int npts, int role, int fmt, float att_eps, const int* u_slot, const void* A_in, const void* B7_in,
                    const void* W, float* pool_part, int n_ctas, void* stream);

/* tensor-core (tcgen05 kind::tf32, fp32 accumulate) version of pcreid_sa_edge_mlp: same arguments except that the
 * two weight matrices are fp32 operand images [k/4][n][4] of the (C_out, C_in) BatchNorm-folded weights and that P1 / Cc
 * are POINT-major ((b,n,C) / (b,S,C): a gathered neighbour is one contiguous vector); C in {32, 64, 128}.  Fast mode of the encoder (error ~1e-3 relative: tf32 operands). */
int pcreid_sa_edge_mlp_tc(int B, int C, int N, int S, int k, const float* P1, const float* Cc, const int* idx,
                          const float* W2img, const float* b2, const float* W3img, const float* b3, float* out,
                          int n_ctas, void* stream);

/* Second generation of pcreid_sa_edge_mlp_tc (csrc/sa_tc2.cu): same arithmetic and arguments; producer warps gather
 * relu(P1 + Cc) straight into tensor memory (A operand of GEMM 1), the first accumulator becomes the A operand of GEMM 2
 * in place, max over the k edges by warp redux, P1 of the current object resident in shared memory when it fits.
 * out element (b, c, s) at b*C*S + c*S + s, or with out_pm != 0 point-major at b*S*C + s*C + c.
 * 16 <= k <= 128, C in {32, 64, 128}; else PCREID_ERR_UNSUPPORTED (use pcreid_sa_edge_mlp_tc). */
int pcreid_sa_edge_mlp_tc2(int B, int C, int N, int S, int k, const float* P1, const float* Cc, const int* idx,
                           const float* W2img, const float* b2, const float* W3img, const float* b3, float* out,
                           int out_pm, int n_sms, void* stream);

/* Fused linear-attention blocks of the Point Transformer encoder on the tensor cores (tcgen05 kind::tf32; fast mode;
 * csrc/attn_tc.cu).  Replace the cn_linear / linattn_scale / cn_groupnorm chains of Self_Attention and FP_SA
 * (mmdet3d/models/pointnet2_utils.py:55-114, 362-437).  All weights are fp32 operand images [k/4][n][4] of the
 * (C_out, C_in) torch weights, concatenated into one blob in the order given below; channel counts are multiples of 16
 * (inputs: of 8, zero padded) and at most 128 model channels, else PCREID_ERR_UNSUPPORTED.
 * front: key-side rows:  pos = Wp2 relu(Wp0 xyz + bp0) + bp2;  out[:, 0:NFP] = Wfp (feat + pos);
 *        out[:, NFP:NFP+NF] = Wf feat.   wp0 (3, DP) k-major; blob = [Wp2 (DP->C2)][Wfp (C2->NFP)][Wf (C2->NF)].
 * kv_img: per object and head h the operand image of KV_h = sum_s (elu(k_s)+1) (x) v_s (dh x dh: kvimg is (B', H, dh*dh)
 *        floats, B' = B rounded up to pcreid_attn_back_objects_per_tile) and ksum (B, d) = sum_s (elu(k_s)+1); k, v
 *        channel-major (B, d, S) views (pre-activation).  The reference's v / S and x S cancel and are not applied.
 * back:  query-side rows: q (B, D, rows) given, or q = Wq feat1 when q == NULL;  att_h = (elu(q_h)+1) KV_h / ((elu(q_h)+1).ksum_h + 1e-6);
 *        msg = LayerNorm1(Wm att);  out = LayerNorm2(W2 relu(W0 [feat1 ; msg])) (+ feat1 when res);
 *        blob = [Wq (C1P->D) unless q given][Wm (D->D)][W0a (C1P->2D)][W0b (D->2D)][W2 (2D->CO)], C1P = C1 rounded up to 8;
 *        feat1 channel-major (B, C1, rows) or, with f1_pm, point-major (B, rows, C1). */
int pcreid_attn_front_blob_bytes(int C2, int DP, int NFP, int NF);
int pcreid_attn_front(int B, int S, int C2, int DP, int NFP, int NF, const float* xyz, const float* feat, long long f_bs, int ldf,
                      const float* wp0, const float* bp0, const float* bp2, const void* blob, float* out, long long o_bs, int ldo,
                      void* stream);
int pcreid_linattn_kv_img(int B, int S, int d, int H, const float* K, long long k_bs, int ldk, const float* V, long long v_bs, int ldv,
                          float* kvimg, float* ksum, void* stream);
int pcreid_attn_back_objects_per_tile(int rows, int D);
int pcreid_attn_back_blob_bytes(int D, int C1P, int CO, int qpre);
int pcreid_attn_back(int B, int rows, int D, int H, int C1, int CO, int res, int f1_pm, const float* feat1, long long f1_bs,
                     int ldf1, const float* q, long long q_bs, int ldq, const float* ksum, const float* kvimg, const float* g1,
                     const float* b1, const float* g2, const float* b2, const void* blob, float* out, long long o_bs, int ldo,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PCREID_H_ */
