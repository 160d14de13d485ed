/*
 * p2s_b200.h -- C ABI of libp2s_b200.so, the B200 (sm_100a) implementation of the Points2Surf
 * SDF-inference hot path (SURVEY.md section 8).  Plain pointers and sizes only; no torch types.
 *
 * The reference (ErlerPhilipp/points2surf) is pure Python, so "the FFI a maintainer would bind" is
 * a ctypes stub; INTEGRATION.md shows it.  Each entry point names the reference interface it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; p2s_last_error() gives the message
 *     (thread-local, valid until the next call on the same thread).
 *   - `*_dev` functions take DEVICE pointers on the model's device and enqueue on `stream`
 *     (a cudaStream_t passed as void*; NULL = default stream).  They do not synchronise unless
 *     documented ("sync: count read-back").  Functions without a model run on the calling thread's
 *     current CUDA device, which must be the device of their pointers and of `stream`.
 *   - `*_host` functions take HOST pointers, perform H2D/D2H copies on the model's internal stream
 *     and return after the result is in the host buffer.
 *   - all float data is IEEE fp32, all index data int32, row-major, densely packed.
 *   - there is no CPU fallback anywhere behind this ABI.
 */
#ifndef P2S_B200_H
#define P2S_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P2S_ABI_VERSION 2

/* ------------------------------------------------------------------ library / errors ----------- */
int p2s_abi_version(void);
const char* p2s_last_error(void);
/* number of kernels this library has launched since load / since the last reset (bench.py's
 * gpu_launches claim is read from here). */
uint64_t p2s_launch_count(void);
void p2s_launch_count_reset(void);

/* ------------------------------------------------------------------ model ---------------------- */
typedef struct p2s_model p2s_model;

/* Mirrors the constructor arguments of source/points_to_surf_model.py:238-240 as used by
 * source/points_to_surf_eval.py:150-166.  Supported subset (SURVEY.md section 8b): sym_op='max',
 * single_transformer=0, use_feat_stn=1, output_dim=2 (imp_surf_magnitude, imp_surf_sign). */
typedef struct {
    int32_t use_point_stn;      /* train_opt.use_point_stn                                  */
    int32_t shared_transformer; /* train_opt.shared_transformer                             */
    int32_t points_per_patch;   /* train_opt.points_per_patch (300)                         */
    int32_t sub_sample_size;    /* train_opt.sub_sample_size (1000)                         */
    int32_t net_size;           /* train_opt.net_size (1024; must be 1024 for the TC path)  */
} p2s_model_config;

/* Weight blob: BatchNorm (eval mode, eps 1e-5) already folded into the preceding Conv1d/Linear
 * (w' = w*g/sqrt(var+eps), b' = (b-mean)*g/sqrt(var+eps)+beta), every layer stored as
 * W[Cout][Cin] row-major followed by b[Cout], layers concatenated in this order:
 *   STN3(p)  := p.conv1 p.conv2 p.conv3 p.fc1 p.fc2 p.fc3            (QSTN, fc3 -> 4)
 *   STN64(p) := p.conv1 p.conv2 p.conv3 p.fc1 p.fc2 p.fc3            (STN dim 64, fc3 -> 4096)
 *   FEAT(p, qstn) := [STN3(p.stn1) if qstn] STN64(p.stn2) p.conv0a p.conv0b p.conv1 p.conv2 p.conv3
 *   blob := [STN3(point_stn) if use_point_stn && shared_transformer]
 *           FEAT(feat_local, 0)  FEAT(feat_global, use_point_stn && !shared_transformer)
 *           fc1_local fc1_global fc2 fc3 fc4
 * points2surf_b200/weights.py builds it from a reference state_dict. */
size_t p2s_model_blob_floats(const p2s_model_config* cfg);

/* Replaces make_regressor (source/points_to_surf_eval.py:150-171): builds the device-resident,
 * kernel-ready weight set on CUDA device `device`. */
int p2s_model_create(const p2s_model_config* cfg, const float* blob_host, size_t blob_floats,
                     int device, p2s_model** out);
void p2s_model_destroy(p2s_model* m);

/* Arithmetic of the per-point MLP stacks:
 *   P2S_PRECISION_FP32  CUDA-core fp32 FMA everywhere (accuracy path)
 *   P2S_PRECISION_TC    tcgen05 tensor cores, fp16 operands (11-bit significand, same as the TF32 the
 *                       reference's cuDNN Conv1d uses on Ampere+), fp32 accumulate; queries whose
 *                       |sign logit| < guard_band are recomputed on the tensor cores in split precision
 *                       (hi + lo fp16 operands, fp32-level accuracy). */
#define P2S_PRECISION_FP32 0
#define P2S_PRECISION_TC 1
int p2s_model_set_precision(p2s_model* m, int precision, float guard_band);
/* number of queries recomputed in split precision (guard band) since the last call; sync. */
int p2s_model_last_guard_count(p2s_model* m, int64_t* count);

/* Instrumentation for bench.py's roofline: when enabled, every launch of the dominant kernel (the tensor-core
 * PointNet pass) is bracketed by CUDA events on its stream.  p2s_profile_get synchronises on those events and
 * returns the summed device time, the number of launches and their algorithmic FLOPs (un-padded points,
 * SURVEY.md section 8d), then keeps accumulating until the next p2s_profile_enable call. */
int p2s_profile_enable(p2s_model* m, int on);
int p2s_profile_get(p2s_model* m, double* ms, int64_t* launches, double* flops);

/* Diagnostic tap used by the parity tests: when `aux` (device, [B][P2S_AUX_STRIDE] floats) is non-NULL every
 * following forward also writes, per query, the point rotation R (9), feat_local's max feature (1024) and
 * feat_global's max feature (1024) -- trans / the PointNetfeat outputs of points_to_surf_model.py:326-343. */
#define P2S_AUX_STRIDE 2064
int p2s_model_set_debug_aux(p2s_model* m, float* aux);

/* PointsToSurfModel.forward (source/points_to_surf_model.py:296-352), eval mode.
 *   patch_pts_ps            [B, points_per_patch, 3]   x['patch_pts_ps']
 *   pts_sub_sample_ms       [B, sub_sample_size, 3]    x['pts_sub_sample_ms'] (model space, NOT yet centred;
 *                                                       unlike the reference this op does not modify it)
 *   imp_surf_query_point_ms [B, 3]                     x['imp_surf_query_point_ms']
 *   logits                  [B, 2]                     (|d| logit, sign logit) */
int p2s_forward_dev(p2s_model* m, const float* patch_pts_ps, const float* pts_sub_sample_ms,
                    const float* imp_surf_query_point_ms, int64_t B, float* logits, void* stream);
int p2s_forward_host(p2s_model* m, const float* patch_pts_ps, const float* pts_sub_sample_ms,
                     const float* imp_surf_query_point_ms, int64_t B, float* logits);

/* post_process + combine (source/sdf_nn.py:11-21, source/points_to_surf_eval.py:184-196,263-271,205-207):
 * sdf = tanh(l0)^2 * radius * (l1 >= 0 ? +1 : -1), NaN -> 1.  patch_radius_ms == NULL is the fixed-radius case
 * (train_opt.patch_radius > 0): the magnitude is not rescaled (points_to_surf_eval.py:188-189,364-368). */
int p2s_sdf_from_logits_dev(const float* logits, const float* patch_radius_ms, int64_t B,
                            float* sdf, void* stream);

/* ------------------------------------------------------------------ query assembly ------------- */
/* sdf.get_voxel_centers_grid_smaller_pc (source/sdf.py:46-70): candidate voxels within an eps^3 box
 * of any occupied voxel, last index plane dropped, in np.nonzero (C) order.
 *   pts [N,3] in [-1,1)^3 (points outside are ignored; the reference would raise / wrap)
 *   lin_idx [cap] receives (ix*res+iy)*res+iz ; *count_host the number found (may exceed cap: then
 *   only the first cap are written).  sync: count read-back. */
int p2s_query_grid_dev(const float* pts, int64_t N, int res, int eps, int32_t* lin_idx, int64_t cap,
                       int64_t* count_host, void* stream);
/* volume_space_to_model_space (source/sdf.py:78-79) of the voxel centres, cast to fp32: [Q,3]. */
int p2s_query_points_dev(const int32_t* lin_idx, int64_t Q, int res, float* query_pts_ms, void* stream);

/* point_cloud.get_patch_kdtree in kNN mode + get_patch_radii + model_space_to_patch_space
 * (source/base/point_cloud.py:174-175, source/base/utils.py:62-69,80-88, source/data_loader.py:340-350).
 * Exact: neighbours are the k smallest float64 distances on the float32 coordinates, ascending
 * (cKDTree semantics); radius and normalisation are float32 like NumPy's.
 *   patch_ids [Q,k] (may be NULL)  patch_pts_ps [Q,k,3]  patch_radius_ms [Q] */
int p2s_knn_patch_dev(const float* pts, int64_t N, const float* query_pts_ms, int64_t Q, int k,
                      int32_t* patch_ids, float* patch_pts_ps, float* patch_radius_ms, void* stream);

/* point_cloud.get_patch_kdtree in ball-query mode (patch_radius > 0, the radius ablations
 * experiments/train_p2s_{small,medium,large}_radius.sh) + the padding rule and fixed-radius normalisation of
 * PointcloudPatchDataset.__getitem__ (source/base/point_cloud.py:176-192, source/data_loader.py:340-350):
 * every point with float64 distance <= patch_radius (cKDTree.query_ball_point on the float32 coordinates); when there are
 * more than k, a uniformly random k-subset without replacement (the reference's rng.choice; here the k smallest
 * Philox clocks keyed by (seed, query index): same law, different stream, independent of batching); when there are fewer,
 * the patch is padded with the query point (patch-space origin, id 0 like the reference's -1 -> 0).
 *   patch_ids [Q,k] (may be NULL; ascending id when nothing is dropped)  patch_pts_ps [Q,k,3] = (p - q) / patch_radius
 *   patch_radius_ms [Q] = patch_radius   in_ball_counts [Q] (may be NULL) = points found before sub-setting / padding */
int p2s_ball_patch_dev(const float* pts, int64_t N, const float* query_pts_ms, int64_t Q, int64_t query_index_base,
                       int k, double patch_radius, uint64_t seed, int32_t* patch_ids, float* patch_pts_ps,
                       float* patch_radius_ms, int32_t* in_ball_counts, void* stream);

/* utils.get_point_cloud_sub_sample (source/base/utils.py:196-227), N >= sub_sample_size.
 *   mode P2S_SUBSAMPLE_UNIFORM : with replacement, like rng.randint             (utils.py:213-216)
 *   mode P2S_SUBSAMPLE_WEIGHTED: without replacement, p ~ clip(1-1.5 d/dmax, .05, 1) (utils.py:200-208,218-219)
 * Counter-based Philox4x32-10 keyed by (seed, query index): results do not depend on batch
 * partitioning or GPU count.  Same distribution as the reference, not the same MT19937 stream.
 *   sub_ids [Q,S] */
#define P2S_SUBSAMPLE_WEIGHTED 0
#define P2S_SUBSAMPLE_UNIFORM 1
int p2s_subsample_dev(const float* pts, int64_t N, const float* query_pts_ms, int64_t Q,
                      int64_t query_index_base, int S, int mode, uint64_t seed, int32_t* sub_ids,
                      void* stream);
/* pts[sub_ids] -> [Q,S,3] (model space, not centred: what __getitem__ returns, data_loader.py:397). */
int p2s_gather_points_dev(const float* pts, const int32_t* ids, int64_t count, float* out, void* stream);

/* ------------------------------------------------------------------ fused reconstruction ------- */
/* The eval loop of source/points_to_surf_eval.py:337-404 in reconstruction mode for ONE shape:
 * candidate grid -> per query (kNN patch, sub-sample, network, post-process) -> SDF band.
 *   pts [N,3] device;  on return *Q_host queries, lin_idx [cap] and sdf [cap] device arrays filled
 *   (what the reference writes to rec/query_pts_ms and rec/dist_ms).  first_query/num_queries
 *   select a contiguous slab of the ordered query list (multi-GPU tile sharding); pass 0,-1 for all.
 * sync: count read-back. */
typedef struct {
    int32_t res;              /* --query_grid_resolution */
    int32_t eps;              /* --epsilon               */
    int32_t subsample_mode;   /* train_opt.uniform_subsample ? UNIFORM : WEIGHTED */
    int32_t batch;            /* queries per network batch (0 = library default) */
    uint64_t seed;            /* --seed                  */
    float patch_radius;       /* train_opt.patch_radius: <= 0 kNN patches, > 0 ball-query patches of this radius */
    int32_t reserved;         /* must be 0 */
} p2s_recon_config;
int p2s_reconstruct_dev(p2s_model* m, const p2s_recon_config* rc, const float* pts, int64_t N,
                        int64_t first_query, int64_t num_queries,
                        int32_t* lin_idx, float* sdf, int64_t cap, int64_t* Q_host, void* stream);
int p2s_reconstruct_host(p2s_model* m, const p2s_recon_config* rc, const float* pts_host, int64_t N,
                         int32_t* lin_idx_host, float* sdf_host, int64_t cap, int64_t* Q_host);

/* ------------------------------------------------------------------ volume -> mesh ------------- */
/* add_samples_to_volume + propagate_sign + clamp (source/sdf.py:82-111,114-178,200-202) for the
 * reconstruction case (one sample per voxel).  vol [res^3] fp32 (the reference's float64 volume holds
 * only fp32 distances and -1/0/+1, so fp32 is exact).  *iterations_host = propagation iterations run.
 * sync: convergence flag read-back every few iterations. */
int p2s_sdf_to_volume_dev(const int32_t* lin_idx, const float* sdf, int64_t Q, int res, int sigma,
                          float certainty_threshold, float* vol, int* iterations_host, void* stream);

/* marching cubes at level 0 + unit-cube transform + orientation fix (source/sdf.py:211-227).
 *   verts [vcap,3] fp32 in model space, faces [fcap,3] int32; counts returned on the host.
 * sync: count read-back. */
int p2s_marching_cubes_dev(const float* vol, int res, float level, float* verts, int64_t vcap,
                           int32_t* faces, int64_t fcap, int64_t* nverts_host, int64_t* nfaces_host,
                           void* stream);

/* ------------------------------------------------------------------ mesh acceptance metric ----- */
/* Area-weighted surface sampling (the sampler behind _chamfer_distance_single_file / _hausdorff_distance_single_file,
 * source/base/evaluation.py:229-238; trimesh.sample.sample_surface without the "even" rejection step -- trimesh is
 * absent, parity unpinned).  verts [V,3] fp32, faces [F,3] int32 -> samples [n,3] fp32, face_ids [n] int32 or NULL.
 * Philox stream keyed by (seed, sample index).  async. */
int p2s_mesh_sample_dev(const float* verts, int64_t V, const int32_t* faces, int64_t F, int64_t n,
                        uint64_t seed, float* samples, int32_t* face_ids, void* stream);

/* Exact nearest neighbour of every a[i] in b (cKDTree.query(a, 1), source/base/evaluation.py:246-250): dist [na]
 * fp32 Euclidean distance, idx [na] int32 (lowest index on ties); either output may be NULL.  async. */
int p2s_nn_distance_dev(const float* a, int64_t na, const float* b, int64_t nb, float* dist, int32_t* idx,
                        void* stream);

/* Both directed sums and maxima of the nearest-neighbour distances between two sample sets:
 * out4_host = { sum a->b, sum b->a, max a->b, max b->a }.  Chamfer (evaluation.py:252-254) = out[0] + out[1];
 * directed Hausdorff (evaluation.py:301-303) = out[2], out[3].  sync: result read-back. */
int p2s_chamfer_hausdorff_dev(const float* a, int64_t na, const float* b, int64_t nb, double* out4_host,
                              void* stream);

/* ------------------------------------------------------------------ training-step primitives --- */
/* Row a14 (SURVEY.md section 8a): loss + backward + SGD of source/points_to_surf_train.py:441-461,537-563 with the
 * train-mode BatchNorm of source/points_to_surf_model.py.  Activations are row-major [rows, C] fp32.  The host side
 * (points2surf_b200/train.py) sequences these like the reference's autograd graph.  All async on `stream`. */
/* C[z][m][n] = act(sum_k A[z][m][k] W[z][n][k] + bias[n])   (torch conv1d(k=1) / linear / bmm forward) */
int p2s_op_gemm_nt(const float* A, int64_t a_stride_z, int lda, const float* W, int64_t w_stride_z,
                   const float* bias, float* C, int64_t c_stride_z, int ldc, int M, int N, int K, int batch,
                   int relu, void* stream);
/* C[z][n][k] (+)= sum_m A[z][m][n] B[z][m][k]               (weight gradient dW = dZ^T X) */
int p2s_op_gemm_tn(const float* A, int64_t a_stride_z, int lda, const float* B, int64_t b_stride_z, int ldb,
                   float* C, int64_t c_stride_z, int ldc, int M, int N, int K, int batch, int accumulate,
                   void* stream);
/* out[z][c][r] = in[z][r][c] */
int p2s_op_transpose(const float* in, float* out, int rows, int cols, int batch, void* stream);
/* BatchNorm1d(train): s1 = sum x, s2 = sum x^2 over the M rows (f64 [C] each) */
int p2s_op_col_stats(const float* x, int64_t M, int C, double* s1, double* s2, void* stream);
int p2s_op_col_sum(const float* x, int64_t M, int C, double* s1, void* stream);
/* mean, invstd = 1/sqrt(biased var + eps); running stats updated like torch (unbiased var) when non-NULL */
int p2s_op_bn_finalize(const double* s1, const double* s2, int64_t M, int C, float eps, float momentum,
                       float* mean, float* invstd, float* running_mean, float* running_var, void* stream);
/* y = act(gamma (z - mean) invstd + beta) */
int p2s_op_bn_apply(const float* z, int64_t M, int C, const float* mean, const float* invstd,
                    const float* gamma, const float* beta, int relu, float* y, void* stream);
/* dz from dy through act + BatchNorm(train); y = forward output for the ReLU mask or NULL; outputs s1 = dbeta,
 * s2 = dgamma (f64 [C]) */
int p2s_op_bn_backward(const float* dy, const float* z, const float* y, int64_t M, int C, const float* mean,
                       const float* invstd, const float* gamma, double* s1, double* s2, float* dz, void* stream);
/* BatchNorm(train)(+ReLU) fused with the max over the npts points of each query (the conv3 layers): forward from the
 * pre-BN z [B*npts, C] with mean / invstd from p2s_op_col_stats + p2s_op_bn_finalize; backward builds dz directly
 * from dout [B,C] (s1 = dbeta, s2 = dgamma, f64 [C]) */
int p2s_op_bn_maxpool_fwd(const float* z, int64_t B, int npts, int C, const float* mean, const float* invstd,
                          const float* gamma, const float* beta, int relu, float* out, int32_t* arg, void* stream);
int p2s_op_bn_maxpool_bwd(const float* dout, const int32_t* arg, const float* out, const float* z, int64_t B,
                          int npts, int C, const float* mean, const float* invstd, const float* gamma, int relu,
                          double* s1, double* s2, float* dz, void* stream);
/* MaxPool1d over the npts points of each query: y [B, npts, C] -> out [B, C], arg [B, C] (first maximum) */
int p2s_op_maxpool_fwd(const float* y, int64_t B, int npts, int C, float* out, int32_t* arg, void* stream);
int p2s_op_maxpool_bwd(const float* dout, const int32_t* arg, int64_t B, int npts, int C, float* dy, void* stream);
/* compute_loss for outputs (imp_surf_magnitude, imp_surf_sign), source/points_to_surf_train.py:550-561 and
 * source/sdf_nn.py:30-40: loss_out (device f64 [2]) = {w_mag * mse(tanh|p0|, tanh|t/r|), w_sign * bce(p1, s)};
 * dpred [B,2] = gradient of their sum (NULL: forward only).  fixed_radius != 0 skips the division by r. */
int p2s_op_loss(const float* pred, const float* target_mag, const float* radius, const float* target_sign,
                int64_t B, float w_mag, float w_sign, int fixed_radius, double* loss_out, float* dpred,
                void* stream);
/* utils.batch_quat_to_rotmat (source/base/utils.py:13-46) forward and backward.  q4 [B,4] is the raw fc3 output of the
 * QSTN; the identity quaternion (1,0,0,0) is added inside (source/points_to_surf_model.py:124-126).  R, dR [B,9]. */
int p2s_op_quat_to_rot(const float* q4, float* R, int64_t B, void* stream);
int p2s_op_quat_to_rot_bwd(const float* q4, const float* dR, int64_t B, float* dq, void* stream);
/* x[b][:] += v[:]  (identity quaternion / identity matrix offsets) */
int p2s_op_add_row(float* x, const float* v, int64_t B, int C, void* stream);
/* out[b][p][:] = in[b][p][:] - q[b][:]  (source/points_to_surf_model.py:303) */
int p2s_op_center(const float* in, const float* q, int64_t B, int npts, float* out, void* stream);
/* y += a x */
int p2s_op_axpy(float* y, const float* x, float a, int64_t n, void* stream);
/* torch.optim.SGD(momentum) update (source/points_to_surf_train.py:406,461) */
int p2s_op_sgd(float* param, const float* grad, float* momentum_buf, int64_t n, float lr, float momentum,
               int first_step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* P2S_B200_H */
