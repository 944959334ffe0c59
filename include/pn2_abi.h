/*
 * pn2_abi.h -- C ABI of libpn2_b200.so, the B200 (sm_100a) implementation of the
 * PointNet++ set-abstraction / feature-propagation geometry path and the
 * multi-view 2D->3D feature lifting of
 * ChengnanYu/Multi-modal-Learning-on-3D-Point-Clouds.
 *
 * Conventions (mirroring the reference's launcher seam, the *_gpu.h files under utils/src):
 *   - every pointer is a DEVICE pointer into memory the caller owns; outputs
 *     are caller-allocated; nothing is retained between calls;
 *   - tensors are dense, row-major, fp32 / int32 exactly as the reference's;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream); every call only enqueues work on it and returns;
 *   - the return value is a pn2_status.  Unlike the reference (which prints
 *     and calls exit(-1), e.g. utils/src/sampling_gpu.cu:39-43) a failure is
 *     reported to the caller; pn2_last_error() gives the message.
 *
 * Each entry point names the reference interface it replaces.
 */
#ifndef PN2_ABI_H
#define PN2_ABI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PN2_ABI_VERSION 1

typedef enum pn2_status {
    PN2_OK = 0,
    PN2_ERR_INVALID_ARGUMENT = 1, /* bad dims / null pointer / misaligned pointer */
    PN2_ERR_UNSUPPORTED = 2,      /* shape outside what the kernels implement */
    PN2_ERR_CUDA = 3              /* a CUDA runtime call or launch failed */
} pn2_status;

/* Message for the last non-OK status returned on the calling thread ("" if none). */
const char *pn2_last_error(void);
int pn2_abi_version(void);
/* Number of kernel launches this library has enqueued since load (all threads). */
uint64_t pn2_launch_count(void);

/* ---- the nine operators of the reference's `pointnet2_cuda` module -------------------- */

/* furthest_point_sampling_wrapper (utils/src/pointnet2_api.cpp:19, utils/src/sampling.cpp:36-46,
 * launcher utils/src/sampling_gpu.cu:211-253).  xyz (B,N,3) -> idx (B,M) int32, idx[:,0]=0.
 * `temp` is the reference's (B,N) scratch argument; it is neither read nor written here
 * (running minima live in registers) and may be NULL. */
int pn2_furthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int32_t *idx, void *stream);

/* furthest_point_sampling + gather_operation of the picked coordinates in one launch
 * (model/pointnet_util.py:34-35: FPS, gather, and two layout copies).  new_xyz (B,M,3). */
int pn2_fps_gather(int b, int n, int m, const float *xyz, float *temp, int32_t *idx, float *new_xyz, void *stream);

/* gather_points_wrapper (pointnet2_api.cpp:16, sampling.cpp:11-20, sampling_gpu.cu:26-44).
 * points (B,C,N), idx (B,M) -> out (B,C,M) */
int pn2_gather_points(int b, int c, int n, int npoints, const float *points, const int32_t *idx, float *out, void *stream);

/* gather_points_grad_wrapper (pointnet2_api.cpp:17, sampling.cpp:23-33, sampling_gpu.cu:65-83).
 * grad_out (B,C,M), idx (B,M) -> grad_points (B,C,N) += ; caller pre-zeroes grad_points. */
int pn2_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out, const int32_t *idx, float *grad_points, void *stream);

/* ball_query_wrapper (pointnet2_api.cpp:11, ball_query.cpp:14-25, ball_query_gpu.cu:48-62).
 * new_xyz (B,M,3), xyz (B,N,3) -> idx (B,M,nsample).  The whole of idx is written
 * (rows with an empty ball become zeros, as the reference's pre-zeroed buffer gives). */
int pn2_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz, const float *xyz, int32_t *idx, void *stream);

/* group_points_wrapper (pointnet2_api.cpp:13, group_points.cpp:25-36, group_points_gpu.cu:69-83).
 * points (B,C,N), idx (B,npoints,nsample) -> out (B,C,npoints,nsample) */
int pn2_group_points(int b, int c, int n, int npoints, int nsample, const float *points, const int32_t *idx, float *out, void *stream);

/* group_points_grad_wrapper (pointnet2_api.cpp:14, group_points.cpp:11-22, group_points_gpu.cu:28-44) */
int pn2_group_points_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out, const int32_t *idx, float *grad_points, void *stream);

/* three_nn_wrapper (pointnet2_api.cpp:21, interpolate.cpp:14-23, interpolate_gpu.cu:55-74).
 * unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3) SQUARED distances, idx (B,n,3) */
int pn2_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int32_t *idx, void *stream);

/* three_interpolate_wrapper (pointnet2_api.cpp:22, interpolate.cpp:26-39, interpolate_gpu.cu:99-117).
 * points (B,C,m), idx/weight (B,n,3) -> out (B,C,n) */
int pn2_three_interpolate(int b, int c, int m, int n, const float *points, const int32_t *idx, const float *weight, float *out, void *stream);

/* three_interpolate_grad_wrapper (pointnet2_api.cpp:23, interpolate.cpp:41-54, interpolate_gpu.cu:144-161).
 * grad_out (B,C,n) -> grad_points (B,C,m) += ; caller pre-zeroes grad_points. */
int pn2_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int32_t *idx, const float *weight, float *grad_points, void *stream);

/* ---- multi-view lifting (utils/projection.py:166-256, model/pointnet2multiview.py:27-43,80-102) ---- */

#define PN2_REDUCE_MAX 0   /* F.max_pool1d over views, model/pointnet2multiview.py:39 */
#define PN2_REDUCE_FIRST 1 /* first view, later views fill all-zero columns, :93-98 */

/* Per-view parameters of the lifting in one launch (utils/projection.py:25-95 and :178, ~25 torch ops per view in the
 * reference): c2w (num_views,4,4) camera-to-world poses; cam_corners = HOST pointer to 8x3 floats, the camera-space
 * frustum corners depth_to_skeleton(u,v,d) for (u,v) in (0,0),(W-1,0),(W-1,H-1),(0,H-1) x d in (depth_min, depth_max)
 * -> w2c (num_views,4,4) = inverse pose (fp64 adjugate, rounded once), corner2 / corner4 (num_views,3), normals
 * (num_views,6,3), the inputs of pn2_lift_views / pn2_frustum_count. */
int pn2_lift_setup(int num_views, const float *c2w, const float *cam_corners, float *w2c, float *corner2, float *corner4,
                   float *normals, void *stream);

/* One launch for a whole batch of B clouds x V views: frustum test, projection, nearest-pixel
 * (round-half-even) lookup, bounds + depth test, feature fetch and view reduction.
 *   points (B,N,3); feats (B,V,C,H,W); depth (B,V,H,W); w2c (B,V,4,4) = inverse(camera_to_world);
 *   corner2, corner4 (B,V,3) and normals (B,V,6,3) from compute_frustum_corners/normals
 *   (utils/projection.py:25-95); intr[4] = {fx, fy, cx, cy} (host pointer).
 *   out (B,C,N) fp32; pix (B,V,N) int32 = lifted pixel index v*W+u or -1 (may be NULL);
 *   count (B,V) int32 = number of lifted points per view (may be NULL; must be pre-zeroed). */
int pn2_lift_views(int b, int n, int v, int c, int h, int w, const float *points, const float *feats, const float *depth,
                   const float *w2c, const float *corner2, const float *corner4, const float *normals, const float *intr,
                   float depth_min, float depth_max, float accuracy, int reduce, float *out, int32_t *pix,
                   int32_t *count, void *stream);

/* The same operator taking the camera poses directly: c2w (B,V,4,4) camera-to-world and cam_corners (HOST pointer, 8x3
 * floats, as for pn2_lift_setup) replace w2c / corner2 / corner4 / normals; the per-view parameters are derived inside the
 * projection kernel with the arithmetic of pn2_lift_setup (bit-identical), saving a launch per call. */
int pn2_lift_views_poses(int b, int n, int v, int c, int h, int w, const float *points, const float *feats, const float *depth,
                         const float *c2w, const float *cam_corners, const float *intr, float depth_min, float depth_max,
                         float accuracy, int reduce, float *out, int32_t *pix, int32_t *count, void *stream);

/* Backward of pn2_lift_views / pn2_lift_views_poses with respect to feats: the gradient torch autograd gives for the
 * reference's composition (Projection per view, then the view reduction), deterministic.
 *   feats (B,V,C,H,W) as given to the forward; pix (B,V,N) int32 as the forward wrote it; grad_out (B,C,N)
 *   -> grad_feats (B,V,C,H,W), WRITTEN IN FULL (zero where no point contributes; no pre-zeroing).
 *   PN2_REDUCE_MAX: grad_out[b,c,i] goes to the pixel of the first view (in view order) holding the maximum of channel c,
 *     invisible views taking part with 0 (torch's max pooling takes a new maximum only on a strict >); dropped when that
 *     view does not see the point.
 *   PN2_REDUCE_FIRST: the whole column goes to the first view that sees the point with a column that is not all zero;
 *     without one, to view V-1 if it sees the point (the reference's fill loop assigns from V-1 last), else dropped.
 * Contributions to one element are summed in ascending point index in fp32, without atomics: bit-identical from run to
 * run and under CUDA-graph replay.  Temporary storage comes from the stream-ordered allocator; no host synchronisation. */
int pn2_lift_views_grad(int b, int n, int v, int c, int h, int w, const float *feats, const int32_t *pix, int reduce,
                        const float *grad_out, float *grad_feats, void *stream);

/* Best-view selection of the ScanNet loader (data_utils/ScanNetDataLoader.py:87-105 -> utils/projection.py:132-164):
 * number of the n points inside the frustum of each of num_poses cameras, evaluated in fp64 as the reference does.
 * corner2/corner4 (P,3), normals (P,6,3) as for pn2_lift_views; counts (P) int32 must be pre-zeroed. */
int pn2_frustum_count(int n, int num_poses, const float *points, const float *corner2, const float *corner4,
                      const float *normals, int32_t *counts, void *stream);

/* ---- fused set-abstraction / feature-propagation blocks (model/pointnet_util.py:70-221) ---- */

#define PN2_MAX_LAYERS 6

/* A stack of 1x1-conv layers with eval-mode BatchNorm folded in:
 *   y = act(W x + bias),  W (cout, cin) row-major fp32 (device), bias (cout) fp32 (device). */
typedef struct pn2_mlp {
    int num_layers;
    int cin[PN2_MAX_LAYERS];
    int cout[PN2_MAX_LAYERS];
    int relu[PN2_MAX_LAYERS];
    const float *weight[PN2_MAX_LAYERS];
    const float *bias[PN2_MAX_LAYERS];
} pn2_mlp;

#define PN2_ORDER_XYZ_FIRST 0  /* SSG concat, model/pointnet_util.py:41 */
#define PN2_ORDER_FEAT_FIRST 1 /* MSG concat, model/pointnet_util.py:157 */

/* Grouping + shared MLP + max over nsample of one SA scale (model/pointnet_util.py:101-109,
 * 152-166), channel-last activations:
 *   xyz (B,N,3); feat (B,N,D) or NULL (D=0); new_xyz (B,M,3); idx (B,M,K) from pn2_ball_query;
 *   out: element (b, p, ch) at out[(b*M + p)*out_stride + out_offset + ch], ch < cout[last]. */
int pn2_sa_mlp_max(int b, int n, int m, int k, int d, const float *xyz, const float *feat, const float *new_xyz,
                   const int32_t *idx, int order, const pn2_mlp *mlp, float *out, int out_stride, int out_offset,
                   void *stream);

/* Interpolation + skip concat + shared MLP of one FP block (model/pointnet_util.py:200-220),
 * channel-last activations:
 *   feat1 (B,n,D1) or NULL; feat2 (B,m,D2); idx/weight (B,n,3) (ignored when m == 1: the single
 *   coarse feature row is repeated, model/pointnet_util.py:202-203); out (B,n,cout[last]). */
int pn2_fp_mlp(int b, int n, int m, int d1, int d2, const float *feat1, const float *feat2, const int32_t *idx,
               const float *weight, const pn2_mlp *mlp, float *out, void *stream);

/* The group_all SA layer (model/pointnet_util.py:50-67, 101-109): concat + shared MLP + max over ALL n points of each
 * cloud, channel-last:
 *   xyz (B,n,3), feat (B,n,D) or NULL (D=0); row bb*n + i = [xyz[bb,i] | feat[bb,i]] (xyz first, not centred);
 *   out: element (bb, ch) at out[bb*out_stride + out_offset + ch], ch < cout[last]; nothing else of `out` is written.
 * n is any value >= 1.  The tiles of one cloud are combined with an integer atomicMax on the bits of the non-negative
 * pooled values, so the last layer must have a ReLU (else PN2_ERR_UNSUPPORTED); the result is bit-identical from run
 * to run.  The pooled columns are zeroed by a kernel on `stream` first: no host synchronisation, graph capturable.
 * Supported stacks: those pn2_mlp_fp32_supported(mlp, 3 + D, 0) accepts (the same row tiles and shared memory layout). */
int pn2_sa_all_mlp_max(int b, int n, int d, const float *xyz, const float *feat, const pn2_mlp *mlp, float *out,
                       int out_stride, int out_offset, void *stream);

/* 1 if pn2_sa_mlp_max (nsample >= 1) / pn2_fp_mlp and pn2_sa_all_mlp_max (nsample == 0) supports this stack fed with c0
 * input channels (layer count, nsample a power of two <= 128, widths within shared memory); 0 otherwise.  No CUDA call. */
int pn2_mlp_fp32_supported(const pn2_mlp *mlp, int c0, int nsample);

/* ---- the shared-MLP layer in TRAINING mode (BatchNorm with batch or running statistics; model/pointnet_util.py:105-107,
 * 162-165,218-220 under autograd), fp32, channel-last row matrices (rows x channels).  See csrc/train_mlp.cu for the algebra. ----
 * forward: z (rows,cout) = act_in(x) W^T + bias, act_in(v) = relu(in_scale v + in_shift) per input channel (the previous
 *   layer's BatchNorm + ReLU; NULL/NULL = identity), w (cout,cin); stats (2,cout) float64, PRE-ZEROED: += sum_r z, sum_r z^2.
 *   stats NULL: no statistics are reduced (a layer whose BatchNorm uses its running statistics), z only. */
int pn2_train_linear_fwd(long long rows, int cin, int cout, const float *x, const float *in_scale, const float *in_shift,
                         const float *w, const float *bias, float *z, double *stats, void *stream);
/* Per-channel BatchNorm quantities from the forward sums (one tiny launch): scale = gamma rstd, shift = beta - mean scale
 * (fp32, the next layer's act_in), mean_rstd (2,c) float64 for the backward; running_mean / running_var (may both be NULL)
 * are updated like torch.nn.BatchNorm in training mode (momentum, unbiased variance). */
int pn2_train_bn_finalize(long long rows, int c, const double *stats, const float *gamma, const float *beta, double eps,
                          double momentum, float *scale, float *shift, double *mean_rstd, float *running_mean,
                          float *running_var, void *stream);
/* Coefficients of dz = ca dy + cb + cc z from the backward sums: coef (3,c) = ca | cb | cc; dgamma (c), dbeta (c). */
int pn2_train_bn_bwd_coeffs(long long rows, int c, const double *sums, const double *mean_rstd, const float *gamma, float *coef,
                            float *dgamma, float *dbeta, void *stream);
/* A BatchNorm that normalises with its RUNNING statistics (eval mode; torch uses batch statistics iff bn.training or no
 * running statistics): scale = gamma rstd, shift = beta - running_mean scale with rstd = 1 / sqrt(running_var + eps) (fp32,
 * the same roles as pn2_train_bn_finalize's), mean_rstd (2,c) float64 = (running_mean, rstd) for the backward.  Writes
 * nothing else: the running statistics are read only. */
int pn2_train_bn_running(int c, const float *running_mean, const float *running_var, const float *gamma, const float *beta,
                         double eps, float *scale, float *shift, double *mean_rstd, void *stream);
/* Its backward from the sums of pn2_train_bn_bwd_reduce (S1 = sum dy, S2 = sum dy z): coef (3,c) = scale | 0 | 0 (dz = scale dy),
 * dgamma = rstd (S2 - running_mean S1), dbeta = S1, dbias = scale S1 (the conv bias gradient, sum_r dz). */
int pn2_train_bn_running_bwd_coeffs(int c, const double *sums, const double *mean_rstd, const float *scale, float *coef,
                                    float *dgamma, float *dbeta, float *dbias, void *stream);
/* a (rows,c) = relu(scale z + shift): the materialised output of the last layer of a stack. */
int pn2_train_bn_relu(long long rows, int c, const float *z, const float *scale, const float *shift, float *a, void *stream);
/* BatchNorm backward reductions: dy = g [scale z + shift > 0]; sums (2,c) float64, PRE-ZEROED: += sum_r dy, sum_r dy z. */
int pn2_train_bn_bwd_reduce(long long rows, int c, const float *g, const float *z, const float *scale, const float *shift,
                            double *sums, void *stream);
/* backward of one layer: dz = ca dy + cb + cc z (per output channel); g_in (rows,cin) = dz W (NULL = not needed; wt = W^T,
 * (cin,cout) row-major); dw (cout,cin), PRE-ZEROED, += dz^T act_in(x) (fp32 atomics: accumulation order unspecified, as in
 * the reference's backward kernels). */
int pn2_train_linear_bwd(long long rows, int cin, int cout, const float *x, const float *in_scale, const float *in_shift,
                         const float *wt, const float *g, const float *z, const float *scale, const float *shift,
                         const float *ca, const float *cb, const float *cc, float *g_in, float *dw, void *stream);

/* ---- first and last layer of a whole training-mode SA scale / FP block: the grouped or interpolated operand is read
 * where it lies and never materialised, the pooled output is written without the (rows,c) activation. ----
 * Row source of the first layer (fp32, channel-last, contiguous):
 *   PN2_ROWS_GROUPED (SA): xyz (b,n,3), feat (b,n,d) or NULL (d == 0), new_xyz (b,m,3), idx (b,m,k) in [0,n);
 *     row (bb*m + s)*k + j = [xyz[p] - new_xyz[s] | feat[p]] (PN2_ORDER_XYZ_FIRST) or [feat[p] | xyz[p] - new_xyz[s]]
 *     (PN2_ORDER_FEAT_FIRST), p = idx[bb,s,j]; the centring is one fp32 subtraction.  rows = b*m*k, cin = 3 + d.
 *   PN2_ROWS_INTERP (FP): skip (b,n,d_skip) or NULL (d_skip == 0), feat (b,m,d), idx / weight (b,n,3);
 *     row bb*n + i = [skip[i] | fma(w2,f[i2],fma(w0,f[i0],w1*f[i1]))] (three_interpolate's order); with m == 1 idx and
 *     weight are NULL and the one coarse row is repeated.  rows = b*n, cin = d_skip + d.
 *   PN2_ROWS_ALL (group_all SA): xyz (b,n,3), feat (b,n,d) or NULL (d == 0); row bb*n + i = [xyz[bb,i] | feat[bb,i]]
 *     (not centred).  rows = b*n, cin = 3 + d. */
#define PN2_ROWS_GROUPED 1
#define PN2_ROWS_INTERP 2
#define PN2_ROWS_ALL 3
typedef struct pn2_rows {
    int kind;
    int order; /* PN2_ROWS_GROUPED: PN2_ORDER_XYZ_FIRST or PN2_ORDER_FEAT_FIRST */
    int b, n, m, k, d, d_skip;
    const float *xyz, *new_xyz, *feat, *skip;
    const int32_t *idx;
    const float *weight;
} pn2_rows;
/* pn2_train_linear_fwd with the first layer's operand read from `src` (no act_in). */
int pn2_train_linear_fwd_rows(long long rows, int cin, int cout, const pn2_rows *src, const float *w, const float *bias,
                              float *z, double *stats, void *stream);
/* pn2_train_linear_bwd of the first layer with x read from `src`.  g_in (rows, cin) (NULL = not needed); for
 * PN2_ROWS_INTERP the first d_skip columns go to g_skip (rows, d_skip) and g_in holds the d interpolated columns
 * (rows, d); either may be NULL.  For PN2_ROWS_ALL a row is a point: g_in is the feature gradient (b, n, d) itself
 * (NULL when d == 0) and the xyz columns get no gradient. */
int pn2_train_linear_bwd_rows(long long rows, int cin, int cout, const pn2_rows *src, const float *wt, const float *g,
                              const float *z, const float *scale, const float *shift, const float *ca, const float *cb,
                              const float *cc, float *g_in, float *g_skip, float *dw, void *stream);
/* Last layer + max over the k rows of each of `groups` groups: a = relu(scale z + shift) (as pn2_train_bn_relu), z (groups*k, c);
 * out[gr*out_stride + out_offset + ch] = max_j a, arg (groups, c) uint8 = the first j holding it.  k <= 256. */
int pn2_train_bn_relu_max(long long groups, int k, int c, const float *z, const float *scale, const float *shift, float *out,
                          int out_stride, int out_offset, uint8_t *arg, void *stream);
/* Backward of the pooling: g (groups*k, c) written in full, g = gp[gr*gp_stride + gp_offset + ch] on row j == arg, 0 elsewhere. */
int pn2_train_max_bwd(long long groups, int k, int c, const float *gp, int gp_stride, int gp_offset, const uint8_t *arg,
                      float *g, void *stream);
/* The same pooling over all k >= 1 rows of each group (group_all: a group is a cloud, k its points): out as above, arg
 * (groups, c) int32 = the first row holding the maximum (torch.max(dim)'s index).  Row ranges of one group are combined
 * by a 64-bit atomicMax on (value bits, ~row), exact and independent of the order of the CTAs; out and arg are written
 * in full.  Temporary storage comes from the stream-ordered allocator; no host synchronisation. */
int pn2_train_bn_relu_max_all(long long groups, long long k, int c, const float *z, const float *scale, const float *shift,
                              float *out, int out_stride, int out_offset, int32_t *arg, void *stream);
/* Its backward: g (groups*k, c) written in full, g = gp[gr*gp_stride + gp_offset + ch] on row arg[gr, ch], 0 elsewhere. */
int pn2_train_max_bwd_all(long long groups, long long k, int c, const float *gp, int gp_stride, int gp_offset,
                          const int32_t *arg, float *g, void *stream);

/* ---- the same two blocks on the tcgen05 tensor cores: bf16 operands, fp32 accumulation in TMEM ----
 * Outputs agree with the fp32 entry points within bf16 rounding (2e-2 relative).  Weights are packed once
 * (bf16, pre-swizzled UMMA tiles) with pn2_mlp_pack_bf16; biases are still read from `mlp`.
 *
 * first_layer_rotate: the kernels build the first operand as [features | centred xyz] (SA) or
 * [interpolated | skip] (FP); packing rotates the first layer's weight columns to match:
 *   SA with PN2_ORDER_XYZ_FIRST weights -> 3 (0 when d == 0);  PN2_ORDER_FEAT_FIRST -> 0;  FP -> d1. */
int pn2_mlp_bf16_supported(const pn2_mlp *mlp);       /* 1 if the widths fit shared memory / TMEM */
long long pn2_mlp_pack_bf16_size(const pn2_mlp *mlp); /* bytes of the packed image (16-byte aligned buffer) */
int pn2_mlp_pack_bf16(const pn2_mlp *mlp, int first_layer_rotate, void *packed, void *stream);
/* flags: activations that only travel between tensor-core blocks may be stored as bf16 (they are rounded to bf16 for
 * the MMA operand anyway; for SA gathers the result is bit-identical).  The pointer types below stay `float *`; with a
 * flag set the buffer holds bf16 elements of the same logical shape. */
#define PN2_FLAG_IN_BF16 1   /* SA: feat, FP: feat2 (needs d resp. d2 % 8 == 0, 16-byte aligned rows) */
#define PN2_FLAG_SKIP_BF16 2 /* FP: feat1 (needs PN2_FLAG_IN_BF16 and d1 % 8 == 0) */
#define PN2_FLAG_OUT_BF16 4  /* out */
#define PN2_FLAG_OUT_ARGMAX 8 /* FP only: out is (B,n) uint8, the index of the largest output channel of each row (first
                               * maximum, as numpy.argmax) -- the per-point class prediction the reference's evaluation
                               * loop takes from the logits on the host (train_scannet_semseg.py:204-205).  <= 256 channels. */
int pn2_sa_mlp_max_bf16(int b, int n, int m, int k, int d, const float *xyz, const float *feat, const float *new_xyz,
                        const int32_t *idx, const pn2_mlp *mlp, const void *packed, float *out, int out_stride,
                        int out_offset, int flags, void *stream);
/* row_perm (B,n) int32 or NULL: processing order of the rows of each cloud (a permutation, e.g. the `order` of
 * pn2_grid_build); the result is the same, a spatially coherent order makes the 3-row gather cache friendly. */
int pn2_fp_mlp_bf16(int b, int n, int m, int d1, int d2, const float *feat1, const float *feat2, const int32_t *idx,
                    const float *weight, const pn2_mlp *mlp, const void *packed, const int32_t *row_perm, float *out,
                    int flags, void *stream);

/* three_nn followed by the reference's weight computation (model/pointnet_util.py:205-208):
 * dist = sqrt(dist2); clamp 1e-10; w = 1/dist; w /= sum.  -> idx (B,n,3), weight (B,n,3) */
int pn2_three_nn_weights(int b, int n, int m, const float *unknown, const float *known, int32_t *idx, float *weight, void *stream);

/* Layout helpers between the reference's channel-first tensors and channel-last activations:
 * in (B,R,Cc) -> out (B,Cc,R) */
int pn2_transpose(int b, int r, int c, const float *in, float *out, void *stream);

/* ---- exact neighbour search through a per-cloud uniform grid (csrc/grid.cu) ----
 * Same results as pn2_ball_query / pn2_three_nn (bit-identical), without the brute-force scan.
 * pn2_grid_build sorts each cloud (n <= pn2_grid_max_points()) by cell:
 *   sorted (B,n,4) fp32 {x,y,z,bits(original index)}, 16-byte aligned; cell_start (B, pn2_grid_table_stride()) int32;
 *   order (B,n) int32 = original index of the i-th sorted point (may be NULL); meta (B,8) words;
 *   cell <= 0 picks a cell size from the bounding box.  For ball queries use cell >= 1.01 * radius. */
int pn2_grid_max_points(void);
int pn2_grid_table_stride(void);
int pn2_grid_build(int b, int n, const float *xyz, float cell, float *sorted, int32_t *cell_start, int32_t *order,
                   float *meta, void *stream);
int pn2_ball_query_grid(int b, int n, int m, float radius, int nsample, const float *new_xyz, const float *xyz,
                        const float *sorted, const int32_t *cell_start, const float *meta, int32_t *idx, void *stream);
/* grid over the KNOWN set (m points); query_order (B,n) optional processing order of the unknown points;
 * dist2 (squared) and weight (model/pointnet_util.py:205-208) are optional outputs. */
int pn2_three_nn_grid(int b, int n, int m, const float *unknown, const float *known, const float *sorted,
                      const int32_t *cell_start, const float *meta, const int32_t *query_order, float *dist2,
                      int32_t *idx, float *weight, void *stream);

/* ---- deterministic backwards (SURVEY 8f N1) ----
 * The three reference backwards above accumulate with atomicAdd, so the fp32 summation order changes from run to run.
 * These two calls give the same gradients with a FIXED order (ascending source position) and no atomics.
 * pn2_inverse_index: idx (b,j) int32 with values in [0,n) -> seg_start (b*n + 1) int32 and pos (b,j) int32: the source
 * positions p of cloud `bb` whose idx == k are pos[bb*j + seg_start[bb*n + k] - bb*j ...]: precisely, slots
 * seg_start[bb*n + k] .. seg_start[bb*n + k + 1] of the flattened `pos` hold them in ascending order.  One stable
 * device radix sort; temporary storage comes from the stream-ordered allocator.
 * pn2_scatter_rows_det: grad_points (b,c,n) += sum over those p of weight[bb,p] * grad_out[bb,c,p / div]
 *   gather_points_grad : j = npoints,         div = 1, weight = NULL, grad_out (b,c,npoints)
 *   group_points_grad  : j = npoints*nsample, div = 1, weight = NULL, grad_out (b,c,npoints,nsample)
 *   three_interpolate_grad (n there = m here): j = 3*n_fine, div = 3, weight (b,n_fine,3), grad_out (b,c,n_fine). */
int pn2_inverse_index(int b, int n, long long j, const int32_t *idx, int32_t *seg_start, int32_t *pos, void *stream);
int pn2_scatter_rows_det(int b, int c, int n, long long j, int div, const float *grad_out, const int32_t *seg_start,
                         const int32_t *pos, const float *weight, float *grad_points, void *stream);
/* Channel-last pn2_scatter_rows_det over row matrices, WRITTEN in full (no pre-zeroing; 0 where no row refers to a point):
 *   grad_points[bb,k,c] = sum over the p of (bb,k), ascending, of weight[bb,p] * g_in[(bb*(j/div) + p/div)*row_stride + col_offset + c]
 *   for c < d, grad_points (b,n,d).  SA grouping: j = m*nsample, div = 1, weight NULL; three_interpolate: j = 3*n_fine, div = 3. */
int pn2_scatter_rows_det_cl(int b, int d, int n, long long j, int div, const float *g_in, int row_stride, int col_offset,
                            const int32_t *seg_start, const int32_t *pos, const float *weight, float *grad_points, void *stream);

/* ---- evaluation voxelisation (SURVEY 8f N3) ----
 * utils/pc_util.py:39-51 point_cloud_label_to_surface_voxel_label_fast, as the evaluation loops call it per scene
 * (train_scannet_semseg.py:226-227): over the points of each cloud with mask != 0 (mask NULL = all points),
 * vidx = v0 + v1*nvox0 + v2*nvox0*nvox1 with v = ceil((p - min) / res), nvox = ceil((max - min) / res) in fp32, and
 * numpy.unique(vidx, return_index=True): uvidx (b,n) fp32 ascending, first (b,n) int32 = index of the first point of
 * each voxel, both padded with -1 after count[b] entries; nvox (b,3) fp32 or NULL. */
int pn2_voxel_first_index(int b, int n, const float *xyz, const unsigned char *mask, float res, float *uvidx, int32_t *first,
                          int32_t *count, float *nvox, void *stream);

/* Confusion counters of the evaluation loops (train_scannet_semseg.py:218-223 point-wise, :232-239 voxel-wise), ADDED to
 * out (3, num_classes) int64: [0][l] #(target == l), [1][l] #(target == l and pred == l), [2][l] #(target == l or pred == l).
 * Points: select NULL -> every point i < n with mask[b,i] != 0 (mask NULL = all); voxels: select = `first`, count = `count`
 * of pn2_voxel_first_index.  target (b,n) int64, pred (b,n) uint8 (PN2_FLAG_OUT_ARGMAX output). */
int pn2_label_counts(int b, int n, int num_classes, const int32_t *select, const int32_t *count, const unsigned char *mask,
                     const long long *target, const unsigned char *pred, long long *out, void *stream);

/* ---- whole-scene segmentation (csrc/scene_blocks.cu; the protocol is stated in oracle/whole_scene_ref.py) ----
 * A scene is xyz (n,3) fp32.  Its grid has 1.5 m blocks in x and y from the scene minimum, block id = i * ny + j; a
 * block's segment is the points inside it padded by 0.2 m, in ascending scene index.  Every call only enqueues work;
 * the block counts and chunk counts the caller needs for its allocations are in the device record below, so one
 * evaluation or labelling pass reads back one record.  Not graph-capturable by the caller: output sizes depend on data. */
#define PN2_SCENE_MAX_BLOCKS 65536
typedef struct pn2_scene_grid {
    float cmin[3], cmax[3]; /* per-axis minimum / maximum of the scene */
    int32_t nx, ny;         /* ceil(fp64(fl32(cmax - cmin)) / 1.5) along x / y (0 for a zero extent) */
    int32_t count;          /* kept blocks after pn2_scene_keep, chunks after pn2_scene_chunks */
    int32_t reserved;
} pn2_scene_grid;
/* Grid, bounds and segments: grid (device, written), seg_start (PN2_SCENE_MAX_BLOCKS + 2) int32, pos (4n) int32: the
 * segment of block b is pos[seg_start[b] .. seg_start[b+1]).  n >= 1, 4n < 2^31.  A grid of zero extent or of more than
 * PN2_SCENE_MAX_BLOCKS blocks gets empty segments. */
int pn2_scene_index(int n, const float *xyz, pn2_scene_grid *grid, int32_t *seg_start, int32_t *pos, void *stream);
/* Evaluation blocks: slot s of block b reads segment position ((h >> 32) * count) >> 32, h = splitmix64(seed *
 * 0x9E3779B97F4A7C15 + (b << 32 | s)); a block is kept if it is non-empty and (core slots) / npoints >= 0.01 (fp64), core
 * = inside the block padded by 0.001 m.  kept (PN2_SCENE_MAX_BLOCKS) int32 = kept ids ascending, grid->count = their number. */
int pn2_scene_keep(int npoints, unsigned long long seed, const float *xyz, pn2_scene_grid *grid, const int32_t *seg_start,
                   const int32_t *pos, int32_t *kept, void *stream);
/* The nb kept blocks' samples (nx, ny, nb as read from the grid record; more than PN2_SCENE_MAX_BLOCKS blocks is refused):
 * point_index (nb,npoints) int32 scene indices, points (nb,npoints,3+c) = [xyz | feats] rows, weights (nb,npoints) =
 * labelweights[label] * core (core alone without labelweights; 0 for a label outside [0, num_classes)), target
 * (nb,npoints) int64 = labels (labels, labelweights, target may be NULL). */
int pn2_scene_sample(int nx, int ny, int nb, int npoints, unsigned long long seed, int c, const float *xyz, const float *feats,
                     const long long *labels, const float *labelweights, int num_classes, const pn2_scene_grid *grid,
                     const int32_t *seg_start, const int32_t *pos, const int32_t *kept, int32_t *point_index, float *points,
                     long long *target, float *weights, void *stream);
/* Labelling cover: every non-empty block b splits into k = ceil(count / npoints) chunks, chunk c holding segment positions
 * c, c+k, c+2k, ...  first (PN2_SCENE_MAX_BLOCKS + 1) int32 = first chunk of each block (exclusive scan, ends with the
 * total), grid->count = number of chunks. */
int pn2_scene_chunks(int npoints, pn2_scene_grid *grid, const int32_t *seg_start, int32_t *first, void *stream);
/* The chunks in (block, c) order: sizes (n_chunks) int32 = ceil((count - c) / k), point_index (n_chunks,npoints) int32 with
 * slot s reading position c + k * (s mod size), points (n_chunks,npoints,3+c) rows. */
int pn2_scene_chunk_rows(int nx, int ny, int n_chunks, int npoints, int c, const float *xyz, const float *feats,
                         const pn2_scene_grid *grid, const int32_t *seg_start, const int32_t *pos, const int32_t *first,
                         int32_t *point_index, int32_t *sizes, float *points, void *stream);
/* votes (n,num_classes) int32, written in full: one vote votes[point_index, pred] per slot s < sizes[chunk] (integer
 * atomics: exact, independent of order; predictions >= num_classes are ignored).  labels (n) uint8 or NULL = first
 * maximum of each row, as numpy.argmax.  num_classes <= 256. */
int pn2_scene_votes(int n_chunks, int npoints, const int32_t *point_index, const int32_t *sizes, const uint8_t *pred, int n,
                    int num_classes, int32_t *votes, uint8_t *labels, void *stream);

/* ---- training crops from a resident scene bank (csrc/scene_blocks.cu; the protocol is stated in
 * oracle/scene_crops_ref.py) ----
 * A bank packs s scenes: xyz (n,3) fp32, feats (n,c) fp32, labels (n) int64, offsets (s+1) int64, scene k = rows
 * offsets[k] .. offsets[k+1]).  The library trusts offsets (0 = offsets[0] < offsets[1] < ... < offsets[s] = n): the
 * caller validates them once.  bounds (s,6) fp32 = per-scene [min xyz | max xyz].  n >= 1, n < 2^31. */
int pn2_scene_bank_bounds(int s, long long n, const float *xyz, const long long *offsets, float *bounds, void *stream);
/* One training batch of b crops of npoints, crop i from scene scene_ids[i] (device int32).  The call reads the device
 * counter *step, draws with h = splitmix64(seed * 0x9E3779B97F4A7C15 + step) and increments *step on the stream, so it
 * makes no host read and a captured graph draws the next batch on every replay.  Per crop, try t = 0..9 centres a
 * 1.5 m column (full z range) on the scene point at sample_pos(h, i, 2^31 + t, count); the first try whose 0.2 m padded
 * column is >= 70 % labelled (label > 0) and whose 0.01 m core occupies >= 2 % of its 31 x 31 x 62 voxel keys is
 * taken, else the tenth.  Slot j reads position sample_pos(h, i, j, padded count) of the padded points in ascending
 * scene index.  sample_pos(h, i, j, m) = ((splitmix64(h * 0x9E3779B97F4A7C15 + (i << 32 | j)) >> 32) * m) >> 32.
 * Outputs: point_index (b,npoints) int32 bank rows, points (b,npoints,3+c) [xyz | feats], target (b,npoints) int64
 * labels, weights (b,npoints) fp32 = labelweights[label] * core (core alone when labelweights is NULL; 0 for a label
 * outside [0, num_classes)), center (b) int32 scene-local index of the taken centre, tries (b) int32 in 1..10, valid (b)
 * uint8.  A scene id outside [0, s) cannot be refused without a host read: its crop gets tries = 0, valid = 0, center
 * = -1, point_index = -1 and zero rows, targets and weights.  max_count = the largest scene's point count (scratch of
 * b * max_count int32).  Refused: b < 1, npoints < 1, b * npoints >= 2^31, c < 0, n < 1 or n >= 2^31, s < 1,
 * max_count outside [1, n], null pointers. */
int pn2_scene_crops(int s, long long n, int c, int max_count, const float *xyz, const float *feats, const long long *labels,
                    const long long *offsets, const float *bounds, int b, const int32_t *scene_ids, int npoints,
                    unsigned long long seed, long long *step, const float *labelweights, int num_classes, int32_t *point_index,
                    float *points, long long *target, float *weights, int32_t *center, int32_t *tries, uint8_t *valid,
                    void *stream);

/* ---- proposal layer of the nuScenes detector (SURVEY 8f N4) ----
 * model/pointmaskrcnn.py:233-288 iou_spheres: spheres (x, y, z, r), 16-byte aligned rows -> iou (m,n) fp32, every
 * operation rounded to fp32 in the reference's order. */
int pn2_sphere_iou(int m, int n, const float *spheres_a, const float *spheres_b, float *iou, void *stream);
/* model/pointmaskrcnn.py:290-321 nms, b independent problems of up to n <= 4096 spheres (count_in (b) int32 or NULL = n
 * each): visit by descending score (equal scores: lower index first), keep a sphere and drop every later one whose IoU
 * with it is > threshold.  keep (b,n) int32 = kept indices in selection order, padded with -1; count_out (b) int32. */
int pn2_sphere_nms(int b, int n, const float *spheres, const float *scores, const int32_t *count_in, float threshold,
                   int32_t *keep, int32_t *count_out, void *stream);

/* ---- tuning ---- */
/* Kernel policy of furthest point sampling for 4096 < n <= 8192 points per cloud.  Process-wide; read when a launch is
 * issued (or captured into a CUDA graph).  The sampled indices are identical under every policy.
 *   PN2_FPS_AUTO     a 4-CTA cluster per cloud while 4*b CTAs fit the GPU (lowest latency of a single batch: 0.43 ms for
 *                    8192 -> 1024), else ONE_CTA;
 *   PN2_FPS_ONE_CTA  one 256-thread CTA per cloud (0.54 ms): it occupies b SMs instead of 4*b, which is what counts when
 *                    several batches are in flight (measured: 44.2 k -> 52.2 k scenes/s at the time, profiles/README.md);
 *   PN2_FPS_CLUSTER  always the cluster kernel (also for smaller clouds).
 * Returns the previous policy, or -1 for an unknown value. */
enum { PN2_FPS_AUTO = 0, PN2_FPS_ONE_CTA = 1, PN2_FPS_CLUSTER = 2 };
int pn2_set_fps_policy(int policy);

/* ---- developer hooks (tests / profiling; not part of the operator surface) ---- */
/* pn2_set_fps_policy without the return value (bench.py and the profiling scripts): an unknown value is refused and
 * leaves the policy unchanged. */
void pn2_debug_set_fps_mode(int mode);
/* The next pn2_*_bf16 launch on this thread records clock64() phase stamps of CTA 0 into buf (>= 512 int64, device; MMA issuer stamps from [256]). */
void pn2_debug_set_tc_timestamps(long long *buf);
/* Caps the resident CTAs per SM of the tensor-core MLP kernel (bench.py --tc-max-ctas; default 8 = no cap). */
void pn2_debug_set_tc_max_ctas(int n);
/* Worker warps per 128-row tile of the tensor-core MLP kernel: 4 (up to 4 CTAs per SM), 8 (two warps per TMEM lane
 * quarter splitting the columns, up to 2 CTAs per SM) or 0 = chosen by launch size (default).  Results are identical. */
void pn2_debug_set_tc_workers(int n);
/* What the last pn2_sa_mlp_max_bf16 / pn2_fp_mlp_bf16 call on this thread launched: the kernel build (*name, e.g.
 * "bf16_x4_sa", "f32_w8_fp"; "" when the call launched nothing), its grid and threads per CTA.  Any pointer may be
 * NULL.  Returns 1 if that call launched a kernel, else 0.  Recording changes no launch. */
int pn2_debug_last_tc_launch(const char **name, int *grid, int *threads);
/* Kernel choice of pn2_three_interpolate: 0 automatic, 1 tiled kernels only, 32 the lane-along-channel kernel wherever it
 * applies with 512 threads per CTA, 32 | 256 the same with 256 threads per CTA; any other value is automatic.
 * scripts/interp_sweep.py. */
void pn2_debug_set_interp_mode(int mode);

#ifdef __cplusplus
}
#endif
#endif /* PN2_ABI_H */
