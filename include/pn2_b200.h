/*
 * pn2_b200.h -- C ABI of libpn2_b200.so, the sm_100a PointNet++ SA/FP engine.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  In the reference the
 * native boundary is a set of plain C++ launcher functions called from the
 * TensorFlow OpKernel glue; every pn2_* entry point of the first group below
 * replaces exactly one of them, keeps its argument order and meaning, and adds
 *   - a trailing cudaStream_t (the reference launches on the legacy default
 *     stream and ignores TF's compute stream), passed as void*;
 *   - an int status: 0 on success, a negative PN2_E* code otherwise.  The
 *     reference launchers return void and never check CUDA errors.
 * Conventions kept from the reference: the CALLER owns every buffer (outputs
 * and scratch), all tensors are dense row-major fp32 / int32 DEVICE pointers,
 * nothing is allocated or freed inside the library, no host synchronisation.
 * Difference: the *_grad entry points zero their output themselves (the
 * reference does it in the TF glue: tf_sampling.cpp:236, tf_grouping.cpp:271,
 * tf_interpolate.cpp:477).
 *
 * The library is thread-safe and re-entrant; the only process-wide state is an
 * immutable per-device attribute cache.  No torch types cross this boundary.
 */
#ifndef PN2_B200_H_
#define PN2_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef void *pn2_stream_t; /* cudaStream_t */

enum {
    PN2_OK = 0,
    PN2_EINVAL = -1,       /* bad shape / attribute (reference: OP_REQUIRES InvalidArgument) */
    PN2_ELAUNCH = -2,      /* cudaPeekAtLastError() after launch != cudaSuccess */
    PN2_EUNSUPPORTED = -3, /* size outside what the sm_100a kernels are built for */
    PN2_ENULL = -4         /* required pointer is NULL */
};

int pn2_abi_version(void);
const char *pn2_strerror(int code);
/* last CUDA error string seen by a failing launch on this thread ("" if none) */
const char *pn2_last_cuda_error(void);
/* SM budget of the PERSISTENT kernels (the tensor-core GEMMs launch one CTA per SM): with sms > 0 they size
 * their grids for `sms` SMs and leave the rest of the device to kernels running concurrently on another stream
 * (train_step.py runs the weight-independent sampling / neighbour search of the NEXT batch next to the dense
 * forward pass, the reference overlaps its host-side batch preparation the same way, train.py:134-196).
 * 0 = all SMs.  Process-wide; grid sizes are fixed at launch (and baked into a captured graph).
 * pn2_get_sm_budget returns the SM count the next persistent launch would use. */
int pn2_set_sm_budget(int sms);
int pn2_get_sm_budget(void);

/* ===== group 1: one entry point per reference launcher ======================= */

/* replaces farthestpointsamplingLauncher   tf_ops/tf_sampling.cu:218-221
 * inp (b,n,3) -> out (b,m) int32.  The running minimum distances live in registers (one CTA per
 * cloud up to 8192 points, one thread-block cluster per cloud up to 262144), so temp is not
 * touched on those paths.  It is needed -- (b,n) floats, PN2_ENULL if missing -- only by the
 * streaming fall-back: n > 16384 on a device that cannot schedule the cluster, or n > 262144. */
int pn2_fps(int b, int n, int m, const float *inp, float *temp, int *out, pn2_stream_t s);

/* Same result as pn2_fps, always through the thread-block-cluster kernel (one cluster of up to
 * 16 CTAs per cloud, the cloud resident in their shared memories, candidates exchanged through
 * distributed shared memory).  pn2_fps selects it by itself for large clouds; this entry point
 * exists for tests and benchmarks.  PN2_EUNSUPPORTED when n > 262144 or the device cannot
 * co-schedule the cluster. */
int pn2_fps_cluster(int b, int n, int m, const float *inp, int *out, pn2_stream_t s);

/* EXPERIMENTAL in round 1 (never run on a GPU; tests behind PN2_EXPERIMENTAL=1): pn2_fps_cluster with
 * the per-round cluster barrier replaced by a push + remote-mbarrier handshake.  Same results. */
int pn2_fps_cluster_mb(int b, int n, int m, const float *inp, int *out, pn2_stream_t s);

/* replaces cumsumLauncher                  tf_ops/tf_sampling.cu:208-210
 * inp (b,n) -> out (b,n): row-wise inclusive prefix sum, bit-identical to the reference's
 * blocked scan (same fp32 addition order, see oracle/pn2_oracle.c cumsum_row_ref). */
int pn2_cumsum(int b, int n, const float *inp, float *out, pn2_stream_t s);

/* replaces probsampleLauncher              tf_ops/tf_sampling.cu:212-216
 * inp_p (b,n) weights, inp_r (b,m) uniform numbers in [0,1) -> out (b,m) int32 category
 * indices (inverse CDF).  temp: (b,n) floats of scratch, receives the CDF
 * (tf_sampling.cpp:104-108 allocates the same). */
int pn2_prob_sample(int b, int n, int m, const float *inp_p, const float *inp_r, float *temp,
                    int *out, pn2_stream_t s);

/* replaces gatherpointLauncher             tf_ops/tf_sampling.cu:222-225 */
int pn2_gather_point(int b, int n, int m, const float *inp, const int *idx, float *out,
                     pn2_stream_t s);

/* replaces scatteraddpointLauncher         tf_ops/tf_sampling.cu:226-229 (+memset) */
int pn2_gather_point_grad(int b, int n, int m, const float *out_g, const int *idx, float *inp_g,
                          pn2_stream_t s);

/* replaces queryBallPointLauncher          tf_ops/tf_grouping.cu:138-144
 * xyz1 (b,n,3) data, xyz2 (b,m,3) queries -> idx (b,m,nsample), pts_cnt (b,m).
 * Rows without any hit are written as zeros (the reference leaves them uninitialised). */
int pn2_query_ball_point(int b, int n, int m, float radius, int nsample, const float *xyz1,
                         const float *xyz2, int *idx, int *pts_cnt, pn2_stream_t s);

/* EXPERIMENTAL in round 1 (never run on a GPU; tests behind PN2_EXPERIMENTAL=1): pn2_query_ball_point
 * over a hashed uniform grid with cells of edge `radius` -- identical idx / pts_cnt, work proportional
 * to the ball populations instead of b*m*n.  workspace: caller-owned device scratch of at least
 * pn2_ball_grid_workspace_bytes(b, n) bytes, 16-byte aligned. */
long pn2_ball_grid_workspace_bytes(int b, int n);
int pn2_query_ball_point_grid(int b, int n, int m, float radius, int nsample, const float *xyz1,
                              const float *xyz2, int *idx, int *pts_cnt, void *workspace,
                              long workspace_bytes, pn2_stream_t s);

/* replaces groupPointLauncher              tf_ops/tf_grouping.cu:150-154 */
int pn2_group_point(int b, int n, int c, int m, int nsample, const float *points, const int *idx,
                    float *out, pn2_stream_t s);

/* replaces groupPointGradLauncher          tf_ops/tf_grouping.cu:155-162 (+memset) */
int pn2_group_point_grad(int b, int n, int c, int m, int nsample, const float *grad_out,
                         const int *idx, float *grad_points, pn2_stream_t s);

/* replaces threenn_cpu                     tf_ops/tf_interpolate.cpp:213-243
 * xyz1 (b,n,3) queries, xyz2 (b,m,3) known -> dist (b,n,3) squared fp64->fp32, idx (b,n,3) */
int pn2_three_nn(int b, int n, int m, const float *xyz1, const float *xyz2, float *dist, int *idx,
                 pn2_stream_t s);

/* replaces interpolate_label_with_color_cpu tf_ops/tf_interpolate.cpp:71-115
 * sparse_points (num_sparse,3), sparse_labels (num_sparse), dense_points (num_dense,3) ->
 * dense_labels (num_dense) int32, dense_colors (num_dense,3) uint8: label vote among the knn
 * nearest sparse points (exact fp64 distances, nearest first; the label whose running count
 * first becomes the largest wins) and its colour from the reference's 9-entry table.
 * knn <= 32 (PN2_EUNSUPPORTED beyond).  No sparse point at all -> label -1, colour 0. */
int pn2_interpolate_label_with_color(int num_sparse, int num_dense, const float *sparse_points,
                                     const int *sparse_labels, const float *dense_points,
                                     int *dense_labels, unsigned char *dense_colors, int knn,
                                     pn2_stream_t s);

/* replaces threeinterpolate_cpu            tf_ops/tf_interpolate.cpp:307-330 */
int pn2_three_interpolate(int b, int m, int c, int n, const float *points, const int *idx,
                          const float *weight, float *out, pn2_stream_t s);

/* replaces threeinterpolate_grad_cpu       tf_ops/tf_interpolate.cpp:397-421 (+memset) */
int pn2_three_interpolate_grad(int b, int n, int c, int m, const float *grad_out, const int *idx,
                               const float *weight, float *grad_points, pn2_stream_t s);

/* replaces selectionSortLauncher           tf_ops/tf_grouping.cu:145-149 ("next" scope)
 * dist (b,m,n) -> outi (b,m,n), out (b,m,n): the reference's swap-based partial selection sort, bit for
 * bit -- the first k of each row ascending (ties in the reference's permuted-position order), the rest of
 * the row in the order the swaps leave it.  k > 128 with n > 128: PN2_EUNSUPPORTED. */
int pn2_selection_sort(int b, int n, int m, int k, const float *dist, int *outi, float *out,
                       pn2_stream_t s);

/* Fused k nearest neighbours: knn_point of tf_ops/tf_grouping.py:64-89 (squared-distance matrix (b,m,n)
 * in TF + selectionSortLauncher, tf_grouping.cu:95-136) WITHOUT the matrix: distances are evaluated on the
 * fly in fp32 ((dx*dx + dy*dy) + dz*dz, left to right over the c coordinates), the selection is the
 * reference's (ties included).  xyz1 (b,n,c) data, xyz2 (b,m,c) queries -> val (b,m,k) squared distances,
 * idx (b,m,k).  1 <= k <= min(n, 128). */
int pn2_knn_point(int b, int n, int c, int m, int k, const float *xyz1, const float *xyz2, float *val,
                  int *idx, pn2_stream_t s);

/* ===== group 2: fused layer pieces (no reference launcher; they replace the TF
 * graph ops util/pointnet_util.py and util/tf_util.py string between the custom
 * ops).  Strided variants take a leading dimension ld (in floats) so that
 * concatenations are written in place instead of materialised twice. ========== */

/* sample_and_group body after the ball query (pointnet_util.py:43-54 / :252-260):
 * out[b,j,k,:] = concat(xyz[b,idx]-new_xyz[b,j], points[b,idx]) (xyz_first=1, SSG order)
 *             or concat(points[b,idx], xyz[b,idx]-new_xyz[b,j]) (xyz_first=0, MSG order).
 * points may be NULL (c=0); use_xyz=0 drops the xyz part. */
int pn2_group_concat(int b, int n, int m, int nsample, int c, const float *xyz,
                     const float *new_xyz, const float *points, const int *idx, int xyz_first,
                     int use_xyz, float *out, pn2_stream_t s);
/* same with a padded row pitch: row r of the output starts at out + r*ld (ld >= 3+c floats; the
 * padding is not written).  ld % 4 == 0 makes the rows 16-byte aligned for the TMA tensor maps
 * of pn2_linear_fwd / pn2_linear_wgrad. */
int pn2_group_concat_ld(int b, int n, int m, int nsample, int c, const float *xyz,
                        const float *new_xyz, const float *points, const int *idx, int xyz_first,
                        int use_xyz, float *out, int ld, pn2_stream_t s);
/* gradient of the above w.r.t. points (b,n,c) (zeroed here).  grad_xyz (b,n,3) and
 * grad_new_xyz (b,m,3) are optional (NULL = not needed); when given they are zeroed here. */
int pn2_group_concat_grad(int b, int n, int m, int nsample, int c, const float *grad_out,
                          const int *idx, int xyz_first, int use_xyz, float *grad_points,
                          float *grad_xyz, float *grad_new_xyz, pn2_stream_t s);

/* pointnet_fp_module weights (pointnet_util.py:300-303):
 * w = (1/max(d,1e-10)) / sum_3(1/max(d,1e-10)), IEEE division, rows = b*n */
int pn2_fp_weights(int rows, const float *dist, float *weight, pn2_stream_t s);

/* three_interpolate writing rows of stride ldo (>= c): out[(b*n+j)*ldo + l] */
int pn2_three_interpolate_ld(int b, int m, int c, int n, const float *points, const int *idx,
                             const float *weight, float *out, int ldo, pn2_stream_t s);
int pn2_three_interpolate_grad_ld(int b, int n, int c, int m, const float *grad_out, int ldg,
                                  const int *idx, const float *weight, float *grad_points,
                                  pn2_stream_t s);

/* smallest float T with sqrtf(T) >= radius: the ball-query predicate max(sqrt(d2),1e-20f) < radius
 * is evaluated as !(d2 >= T) (exported for tests). */
float pn2_ball_threshold(float radius);

/* dst[r*ldd + j] (=|+=) src[r*lds + j], j < cols */
int pn2_copy_cols(long rows, int cols, const float *src, int lds, float *dst, int ldd,
                  int accumulate, pn2_stream_t s);

/* ---- shared MLP (tf_util.conv2d / conv1d with 1x1 kernels, tf_util.py:54-204) ----
 * Y[M,N] = f(A)[M,K] * W[K,N] + bias[N],  f(a)[.,k] = a_scale ? act(a*a_scale[k]+a_shift[k]) : a
 * (act = ReLU when a_relu).  f is how the previous layer's BatchNorm+ReLU is applied on the
 * fly.  If stats != NULL, stats[0:N] += column sums of Y, stats[N:2N] += column sums of Y^2
 * (fp64, caller zeroes).  mode: 0 = fp32 SIMT kernel, 1 = tcgen05 3xTF32 kernel, -1 = auto;
 * mode + PN2_GEMM_IMAGE_READY (see pn2_linear_prepare): ws already holds this layer's weight image. */
int pn2_linear_fwd(long M, int K, int N, const float *A, int lda, const float *a_scale,
                   const float *a_shift, int a_relu, const float *W, const float *bias, float *Y,
                   double *stats, void *ws, long ws_bytes, int mode, pn2_stream_t s);

/* pn2_linear_fwd + train-mode BatchNorm finalize in ONE call (tf_util.py:572-581 after :181-191): on the
 * tensor-core path the last CTA of the GEMM turns the column statistics into scale / shift / saved
 * (mean | rstd) and updates the moving statistics (a launch of its own otherwise: 22 per training step);
 * other shapes run the fp32 kernel followed by pn2_bn_train_finalize.  stats (2N doubles) and *counter
 * must be zero on entry; moving_mean / moving_var may both be NULL (statistics frozen). */
typedef struct pn2_bn_finalize {
    const float *gamma, *beta;
    float *moving_mean, *moving_var, *scale, *shift, *saved;
    unsigned *counter;
    float eps, decay;
    int unbiased_moving;
} pn2_bn_finalize;
int pn2_linear_fwd_bn(long M, int K, int N, const float *A, int lda, const float *a_scale,
                      const float *a_shift, int a_relu, const float *W, const float *bias, float *Y,
                      double *stats, const pn2_bn_finalize *fin, void *ws, long ws_bytes, int mode,
                      pn2_stream_t s);

/* bytes of caller-owned scratch the tensor-core path of pn2_linear_fwd / pn2_linear_dgrad needs
 * for a K x N layer (the pre-split, pre-swizzled 3xTF32 weight image).  ws may be NULL: the
 * exact fp32 CUDA-core kernel is used then. */
long pn2_linear_workspace_bytes(int K, int N);

/* Weight images built ONCE per optimizer step instead of once per GEMM call: the images of every layer
 * (forward orientation, and dgrad orientation with dgrad=1) are described on the host, the table is
 * copied to the device by the caller, and pn2_linear_prepare builds all of them in ONE launch (after
 * the Adam update).  pn2_linear_fwd / pn2_linear_dgrad then take `mode + PN2_GEMM_IMAGE_READY` and
 * use the image in `ws` as it is.  No reference analogue (cuDNN owns TF's filter transforms). */
#define PN2_GEMM_IMAGE_READY 16
typedef struct pn2_linear_image { /* 64 bytes, opaque to the caller */
    const float *src;
    float *image;
    long s_n, s_k, total;
    int N, Ntot, K, Npad, KC, nchunks;
} pn2_linear_image;
/* bytes of one image (K x N layer; dgrad != 0: the transposed orientation); 0 if the tensor-core path
 * does not cover the shape */
long pn2_linear_image_bytes(int K, int N, int dgrad);
/* fill *out (host memory) for the K x N layer whose weights live at W (device) and whose image will live
 * at image (device, pn2_linear_image_bytes bytes, 128-byte aligned) */
int pn2_linear_image_describe(int K, int N, int dgrad, const float *W, float *image,
                              pn2_linear_image *out);
/* one launch: build the `count` images of the device-resident table */
int pn2_linear_prepare(int count, const pn2_linear_image *table_dev, pn2_stream_t s);

/* dX[M,K] = dY[M,N] * W[K,N]^T */
int pn2_linear_dgrad(long M, int K, int N, const float *dY, const float *W, float *dX, int ldx,
                     void *ws, long ws_bytes, int mode, pn2_stream_t s);

/* dW[K,N] += f(A)[M,K]^T * dY[M,N] ; db[N] += column sums of dY (db may be NULL).
 * Accumulates (split over M with fp32 atomics): caller zeroes dW/db once per step. */
int pn2_linear_wgrad(long M, int K, int N, const float *A, int lda, const float *a_scale,
                     const float *a_shift, int a_relu, const float *dY, float *dW, float *db,
                     int mode, pn2_stream_t s);

/* BatchNorm (tf_util.py:555-581 -> tf.contrib.layers.batch_norm, eps 1e-3).
 * From stats (sum, sumsq over M rows): mean, biased var; scale = gamma*rsqrt(var+eps),
 * shift = beta - mean*scale; saved[0:N] = mean, saved[N:2N] = rstd;
 * moving -= (moving - batch)*(1-decay), the variance fed to the moving average is
 * Bessel-corrected when unbiased_moving != 0 (TF fused kernel, rank-4 inputs). */
int pn2_bn_train_finalize(int N, long M, const double *stats, const float *gamma,
                          const float *beta, float eps, float decay, int unbiased_moving,
                          float *moving_mean, float *moving_var, float *scale, float *shift,
                          float *saved, pn2_stream_t s);
/* inference: scale/shift from the moving statistics */
int pn2_bn_eval_affine(int N, const float *gamma, const float *beta, const float *moving_mean,
                       const float *moving_var, float eps, float *scale, float *shift,
                       pn2_stream_t s);

/* Z[M,N] = act(Y*scale + shift)  (scale/shift NULL = identity) */
int pn2_affine_act(long M, int N, const float *Y, const float *scale, const float *shift,
                   int relu, float *Z, int ldz, pn2_stream_t s);

/* Alternative poolings of pointnet_sa_module (pointnet_util.py:171-191) over X[G*ns,N], the activated
 * output of the shared MLP.  mode 1 "avg" -> out[G,N]; mode 2 "weighted_avg" -> out[G,N] with weights
 * w[G*ns] from pn2_pool_weights (exp(-5 |grouped_xyz|) normalised over nsample, :176-183); mode 3
 * "max_and_avg" -> out[G,2N] = [avg | max] (:187-191) and arg[G,N] = first sample attaining the max.
 * pn2_group_pool_grad: dX[G*ns,N] from dOut (the weights are constants: xyz gradients are dead in the
 * reference's models, model.py feeds xyz as a placeholder). */
int pn2_pool_weights(long G, int ns, const float *grouped_xyz, int ld, float *w, pn2_stream_t s);
int pn2_group_pool(long G, int ns, int N, const float *X, const float *w, int mode, float *out, int *arg,
                   pn2_stream_t s);
int pn2_group_pool_grad(long G, int ns, int N, const float *dOut, const float *w, const int *arg, int mode,
                        float *dX, pn2_stream_t s);

/* Test hook: mask[M,N] (bytes) = 1 where fma(Y, scale, shift) > 0 (Y > 0 without scale/shift) -- the
 * ReLU decision exactly as the prologue / pooling / backward kernels of a chain take it.  Parity tests
 * feed it to the fp64 oracle so that both sides differentiate the same piecewise-linear function. */
int pn2_relu_mask(long M, int N, const float *Y, const float *scale, const float *shift,
                  unsigned char *mask, pn2_stream_t s);

/* out[G,N] = max_{j<ns} act(Y[g*ns+j,:]*scale+shift); arg[G,N] = first j attaining it
 * (pointnet_util.py:167-170 tf.reduce_max over nsample, fused with BN+ReLU) */
int pn2_affine_act_maxpool(long G, int ns, int N, const float *Y, const float *scale,
                           const float *shift, int relu, float *out, int *arg, pn2_stream_t s);

/* Backward of [BN(train) + act] for one layer, dense upstream gradient dZ[M,N]:
 * pass 1: red[0:N] += sum dZh, red[N:2N] += sum dZh*xhat  with dZh = dZ*(z>0 if relu)
 * pass 2: dY = gamma*rstd*(dZh - red0/M - xhat*red1/M); dgamma += red1; dbeta += red0.
 * bn=0 (no BatchNorm): dY = dZh only, pass 1 is skipped by the caller. */
int pn2_bn_bwd_reduce(long M, int N, const float *dZ, int ldz, const float *Y,
                      const float *scale, const float *shift, const float *saved, int relu,
                      double *red, pn2_stream_t s);
int pn2_bn_bwd_apply(long M, int N, const float *dZ, int ldz, const float *Y, const float *scale,
                     const float *shift, const float *saved, const float *gamma, int relu, int bn,
                     const double *red, float *dY, float *dgamma, float *dbeta, pn2_stream_t s);
/* same two passes when the upstream gradient is the max-pooled one: dOut[G,N] routed to arg */
int pn2_bn_bwd_reduce_pool(long G, int ns, int N, const float *dOut, const int *arg,
                           const float *Y, const float *scale, const float *shift,
                           const float *saved, int relu, double *red, pn2_stream_t s);
int pn2_bn_bwd_apply_pool(long G, int ns, int N, const float *dOut, const int *arg,
                          const float *Y, const float *scale, const float *shift,
                          const float *saved, const float *gamma, int relu, int bn,
                          const double *red, float *dY, float *dgamma, float *dbeta,
                          pn2_stream_t s);

/* tf_util.dropout (tf_util.py:646-665): out = keep(i) ? x/keep_prob : 0 with a counter-based
 * generator keyed by (seed, element index); the same call with the same seed regenerates the
 * mask in the backward pass.  seed_dev (optional) is a device-resident increment added to seed, so
 * a captured CUDA graph can draw a fresh mask on every replay.  pn2_dropout_mask exports the mask
 * (0/1 bytes) for tests. */
int pn2_dropout(long n, const float *x, float keep_prob, unsigned long long seed,
                const unsigned long long *seed_dev, float *out, pn2_stream_t s);
int pn2_dropout_mask(long n, float keep_prob, unsigned long long seed, unsigned char *mask,
                     pn2_stream_t s);

/* model.get_loss (model.py:152-161): weighted sparse softmax cross entropy with
 * SUM_BY_NONZERO_WEIGHTS.  acc[0] += sum w*ce, acc[1] += #nonzero w (fp64, caller zeroes);
 * the second call writes loss = acc0/max(acc1,1) and dlogits = g*w*(softmax-onehot)/max(acc1,1)
 * with g = gscale * (gscale_dev ? *gscale_dev : 1) (the upstream gradient, read on the device). */
int pn2_softmax_ce_reduce(long rows, int C, const float *logits, const int *labels,
                          const float *weights, double *acc, pn2_stream_t s);
int pn2_softmax_ce_grad(long rows, int C, const float *logits, const int *labels,
                        const float *weights, const double *acc, float gscale,
                        const float *gscale_dev, float *loss, float *dlogits, pn2_stream_t s);

/* tf.train.AdamOptimizer update on a flat buffer:
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v moments; p -= lr_t*m/(sqrt(v)+eps); gscale multiplies g */
int pn2_adam_step(long n, float *p, const float *g, float *m, float *v, float lr, float beta1,
                  float beta2, float eps, int t, float gscale, pn2_stream_t s);

/* ---- group 2b: whole layers behind one call (SURVEY.md section 8b; no reference analogue) ------------
 * The host side of a layer is native: the entry point walks the op sequence of pointnet_sa_module
 * (util/pointnet_util.py:98-216: ball-query grouping, shared MLP, max pooling -- the configuration model.py
 * uses) or pointnet_fp_module (:285-326) and its exact reverse, launching the kernels declared above on
 * the caller's stream.  Nothing is allocated: every intermediate lives in the caller-owned workspace
 * (pn2_sa_workspace_bytes / pn2_fp_workspace_bytes, 256-byte aligned), and the forward leaves there what the
 * backward needs, so a backward call must see the workspace of its forward call untouched.
 * Layers are described by host arrays of pn2_conv_layer whose pointers are DEVICE arrays owned by the
 * caller: weights W[K,N], bias[N], gamma/beta/moving_mean/moving_var[N] (bn != 0), and for the backward
 * the gradient accumulators dW/dbias/dgamma/dbeta (accumulated into: the caller zeroes them once per step;
 * the bias of a conv that feeds a train-mode BatchNorm gets no gradient: it is exactly zero).
 * xyz gradients are not produced (dead in the reference's models: xyz is a placeholder). */
#define PN2_MAX_LAYERS 8
typedef struct pn2_conv_layer {
    int K, N, bn, relu, rank4; /* rank4: conv2d (Bessel-corrected moving variance), else conv1d */
    const float *W, *bias, *gamma, *beta;
    float *moving_mean, *moving_var; /* updated in place by a training forward; NULL: left alone */
    float *dW, *dbias, *dgamma, *dbeta;
} pn2_conv_layer;
typedef struct pn2_sa_config {
    int b, n, c, npoint, nsample, nlayers, is_training;
    float radius, bn_eps, bn_decay;
} pn2_sa_config;
typedef struct pn2_fp_config {
    int b, n1, n2, c1, c2, nlayers, is_training; /* xyz1 (b,n1,3) dense, xyz2 (b,n2,3) sparse */
    float bn_eps, bn_decay;
} pn2_fp_config;
long pn2_sa_workspace_bytes(const pn2_sa_config *cfg, const pn2_conv_layer *layers);
/* xyz (b,n,3), points (b,n,c) or NULL (c=0) -> new_xyz (b,npoint,3), new_points (b,npoint,N_last),
 * idx (b,npoint,nsample) */
int pn2_sa_forward(const pn2_sa_config *cfg, const pn2_conv_layer *layers, const float *xyz,
                   const float *points, float *new_xyz, float *new_points, int *idx, void *workspace,
                   long workspace_bytes, pn2_stream_t s);
/* d_new_points (b,npoint,N_last) -> parameter gradients (accumulated) and d_points (b,n,c) (may be NULL) */
int pn2_sa_backward(const pn2_sa_config *cfg, const pn2_conv_layer *layers, const float *d_new_points,
                    const int *idx, float *d_points, void *workspace, long workspace_bytes, pn2_stream_t s);
long pn2_fp_workspace_bytes(const pn2_fp_config *cfg, const pn2_conv_layer *layers);
/* points1 (b,n1,c1) or NULL, points2 (b,n2,c2) -> out (b,n1,N_last); concat order [interpolated, points1] */
int pn2_fp_forward(const pn2_fp_config *cfg, const pn2_conv_layer *layers, const float *xyz1,
                   const float *xyz2, const float *points1, const float *points2, float *out,
                   void *workspace, long workspace_bytes, pn2_stream_t s);
int pn2_fp_backward(const pn2_fp_config *cfg, const pn2_conv_layer *layers, const float *d_out,
                    float *d_points1, float *d_points2, void *workspace, long workspace_bytes,
                    pn2_stream_t s);
int pn2_fill_f32(long n, float value, float *dst, pn2_stream_t s);

/* ---- group 3: the input feed in front of the path (SURVEY.md section 8 row f4) ------------------------
 * replaces SemanticFileData.sample() x B + rotate_feature_point_cloud
 *          dataset/semantic_dataset.py:90-186, util/provider.py:72-102, fed at train.py:225-244
 * One launch cuts B fixed-size training samples out of a scene resident in device memory:
 *   points (P,3) fp64 sorted by x (semantic_dataset.py:84-88), colors (P,feat) fp64 or NULL (feat = 0),
 *   labels (P) or NULL, label_weights[num_classes] or NULL (weights default to 1),
 *   center_idx (B): index of each sample's centre point (the caller's RNG, np.random.randint(0, P)),
 *   angles (B) radians about z or NULL (no augmentation), seed: drives the random subset of a box that
 *   holds more than num_point points (key = pn2_box_sample_key(seed, sample, i); the num_point smallest
 *   keys are kept in scene order; a box with fewer points is tiled, :100-106),
 *   scene_z_size = max z - min z of the scene (:131).
 * Outputs: out_data (B,num_point,3+feat) fp32 = [centred (and rotated) xyz | colours], out_labels,
 * out_weights (may be NULL), out_index (B,num_point) scene indices of the sample (the reference's
 * points_raw = points[out_index]), out_count (B) points found in each box.  P < 2^31. */
int pn2_box_sample(int B, long P, int num_point, int feat, const double *points, const double *colors,
                   const int *labels, const float *label_weights, int num_classes,
                   const long *center_idx, const double *angles, double box_size_x, double box_size_y,
                   double scene_z_size, unsigned long long seed, float *out_data, int *out_labels,
                   float *out_weights, int *out_index, int *out_count, pn2_stream_t s);
unsigned pn2_box_sample_key(unsigned long long seed, int sample, long i);

/* ---- group 4: evaluation --------------------------------------------------------------------------------
 * replaces ConfusionMatrix.increment / increment_from_list   util/metric.py:7-83
 *          fed by np.argmax over the host copy of pred        train.py:246-251 (and :307-312, predict.py:90)
 * The logits never leave the device and nothing synchronises the host, so both calls can be captured in a CUDA
 * graph.  cm (C*C, row = ground truth, column = prediction) and skipped are uint64 accumulators the caller
 * zeroes; calls accumulate.  1 <= C <= 128 (PN2_EUNSUPPORTED above). */
/* per row r < rows: pd = arg-max of logits[r, 0:C] with numpy's rule (first maximum; the first NaN wins);
 * if 0 <= labels[r] < C: cm[labels[r]*C + pd] += 1, else *skipped += 1.  pred_out (rows) int32 or NULL. */
int pn2_confusion_from_logits(long rows, int C, const float *logits, const int *labels,
                              unsigned long long *cm, unsigned long long *skipped, int *pred_out,
                              pn2_stream_t s);
/* the same for label pairs; a pair with gt or pd outside [0,C) is skipped (sklearn's
 * confusion_matrix(labels=range(C)), which metric.py:25-30 calls) */
int pn2_confusion_from_labels(long n, int C, const int *gt, const int *pd,
                              unsigned long long *cm, unsigned long long *skipped, pn2_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* PN2_B200_H_ */
