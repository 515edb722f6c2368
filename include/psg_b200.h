/*
 * psg_b200.h -- C ABI of libpsg_b200.so, the B200 (sm_100a) implementation of the PointNet++
 * semantic-segmentation attack hot path of C0ldstudy/PointSecGuard.
 *
 * The reference has no FFI on this path: it is Python over stock PyTorch ops.  Each entry point
 * below therefore names the reference *Python* function(s) it replaces (file:line under
 * /root/reference/PointNet) and is what the torch.library shim in pointsecguard_b200/ops.py binds
 * (see INTEGRATION.md for the reference-side stub a maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - functions enqueue work on `stream` and return immediately; they never synchronise, never
 *     allocate device memory (except psg_net_create / psg_mlp_create, which upload weights once)
 *     and never throw; return value 0 = ok, <0 = PSG_E* below;
 *   - indices are int32 inside the library; the Python layer widens to int64 at the public API;
 *   - "T-layout" is the library's activation layout: float T[rows/128][C/4][128][4], C padded to a
 *     multiple of 16 (pointsecguard_b200/csrc/psg_common.cuh, DESIGN.md section 3).  A T-layout view is passed
 *     as (base pointer, padded width in 16-byte chunks, first chunk of the column slice).
 */
#ifndef PSG_B200_H
#define PSG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSG_OK 0
#define PSG_EINVAL (-1)
#define PSG_EUNSUPPORTED (-2)
#define PSG_EWORKSPACE (-3)
#define PSG_ECUDA (-4)

typedef void *psg_stream_t; /* cudaStream_t */

int psg_version(void);

/* ---- geometric primitives (API layouts: xyz [P,N,3] row-major float32) ----------------------- */

/* farthest_point_sample, pointnet_util.py:63-84.  `start` holds the torch.randint draw of line 75
 * (made by the caller on the CPU generator).  Cloud of problem p is xyz + (p % nclouds) * N * 3, so
 * several problems (attack iterations) may share one cloud.  out_xyz (optional) receives the
 * sampled coordinates = index_points(xyz, fps_idx) of :126.  Kernels by cloud size: N <= 4096 points in registers
 * (one CTA per problem), N <= 16384 in shared memory, N <= 65536 one 8-CTA thread-block cluster per problem (candidates
 * exchanged through distributed shared memory), beyond that a single CTA over a caller-provided min-distance workspace. */
size_t psg_fps_workspace(int P, int N);
int psg_fps(const float *xyz, int nclouds, int P, int N, int npoint, const int32_t *start,
            int32_t *out_idx, float *out_xyz, void *workspace, size_t workspace_bytes, psg_stream_t stream);

/* square_distance, pointnet_util.py:19-40: out[b,i,j] = ((-2 src_i.dst_j) + |src_i|^2) + |dst_j|^2 */
int psg_square_distance(const float *src, const float *dst, int B, int N, int M, float *out, psg_stream_t stream);

/* query_ball_point, pointnet_util.py:87-107; nr = 1 or 2 radii sharing one scan (MSG :246-248). */
int psg_ball_query(const float *xyz, int nclouds, int P, int N, const float *new_xyz, int S, int nr,
                   const double *radius_host, const int *nsample_host, int32_t *out0, int32_t *out1,
                   psg_stream_t stream);

/* Same results as psg_ball_query for every input, bit for bit, through a uniform grid over the cloud
 * (cell edge >= 1.01 r): a centroid tests only the points of its 27 neighbouring cells and emits the hits
 * smallest index first.  A centroid takes the exhaustive scan instead when it has more than 96 hits, or
 * when the distance formula's rounding error, which grows with |q|^2 + max|p|^2, is not proven to stay
 * inside cell^2 - r^2 (clouds far from the origin; the rule is in csrc/ballgrid.cu).  A cloud with a
 * non-finite coordinate is scanned for every centroid, so a NaN distance counts as a hit, as the
 * reference counts it.  ~8x less work than the scan at SA1 densities near the origin. */
size_t psg_ball_grid_workspace(int nclouds, int N);
int psg_ball_query_grid(const float *xyz, int nclouds, int P, int N, const float *new_xyz, int S, int nr,
                        const double *radius_host, const int *nsample_host, int32_t *out0, int32_t *out1,
                        void *workspace, size_t workspace_bytes, psg_stream_t stream);

/* 3-NN + inverse-distance weights, pointnet_util.py:301-307.  w / d2 optional. */
int psg_three_nn(const float *xyz1, int nclouds1, int P, int N, const float *xyz2, int S, int32_t *idx,
                 float *w, float *d2, psg_stream_t stream);

/* index_points, pointnet_util.py:43-60, row-major points [B,N,C], idx int64 [B,M] -> out [B,M,C] */
int psg_index_points(const float *points, const int64_t *idx, int B, int N, int C, int64_t M, float *out,
                     psg_stream_t stream);

/* ---- T-layout building blocks (module-level composition, pointnet_util.py:166-320) ----------- */
int psg_pack_channels_first(const float *x, int64_t sb, int64_t sc, int64_t sn, int B, int C, int N,
                            float *t_base, int t_wchunks, int t_c0, float *xyz_out, psg_stream_t stream);
int psg_unpack_channels_first(const float *t_base, int t_wchunks, int t_c0, int B, int C, int N, float *y,
                              int accumulate, psg_stream_t stream);
/* sample_and_group gather + centre + concat, pointnet_util.py:126-137 / :245-255 (internal column
 * order [features | xyz - centre | 0 pad]) */
int psg_group_points(const float *feats_base, int feats_wchunks, int D, const float *xyz, int nclouds, int Nsrc,
                     const float *new_xyz, const int32_t *idx, int P, int S, int K, float *out_base,
                     int out_cpad, psg_stream_t stream);
int psg_group_max(const float *in_base, int in_wchunks, int64_t groups, int K, int C, float *out_base,
                  int out_wchunks, int out_c0, uint8_t *argmax, psg_stream_t stream);
int psg_group_max_backward(const float *dout_base, int dout_wchunks, int dout_c0, const float *out_base,
                           int out_wchunks, int out_c0, const uint8_t *argmax, int64_t groups, int K, int C,
                           float *dy_base, int dy_wchunks, psg_stream_t stream);
int psg_interpolate(const float *feats_base, int feats_wchunks, int S, const int32_t *idx, const float *w,
                    int64_t P, int N, int ncols, float *out_base, int out_wchunks, int out_c0, psg_stream_t stream);
size_t psg_csr_workspace(int64_t P, int M, int R);
/* pad_group = nsample when `keys` are ball-query rows: slots that repeat the row's first hit
 * (pointnet_util.py:104-106 padding) carry exactly-zero gradient rows and are left out; 0 otherwise */
int psg_csr_build_by_source(const int32_t *keys, int64_t P, int M, int R, int pad_group, int32_t *offsets,
                            int32_t *perm, void *workspace, psg_stream_t stream);
int psg_segment_sum(const float *src_base, int src_wchunks, int src_c0, int64_t src_rows_per_problem, int div,
                    const float *weights, const int32_t *offsets, const int32_t *perm, int M, int R, int64_t P,
                    int ncols, float *dst_base, int dst_wchunks, int dst_c0, int accumulate, psg_stream_t stream);

/* one folded conv(1x1)+BN layer: W [cout][cin] and b [cout] on the HOST; uploads packed copies */
typedef struct psg_mlp psg_mlp;
psg_mlp *psg_mlp_create(const float *w_host, const float *b_host, int cin, int cout);
void psg_mlp_destroy(psg_mlp *m);
/* training: a layer whose W [cout][cin] / b [cout] live in DEVICE memory (nn.Parameter storage) and change every
 * optimiser step; psg_mlp_load (re)packs them into the operand layouts with one small kernel on `stream` */
psg_mlp *psg_mlp_create_device(int cin, int cout);
int psg_mlp_load(psg_mlp *m, const float *w_dev, const float *b_dev, psg_stream_t stream);
/* forward: out = act([a1 | a2] W^T + b), relu = 1/0.  Widths in 16-byte chunks. */
int psg_mlp_forward(const psg_mlp *m, const float *a1_base, int a1_wchunks, int a1_c0, int k1chunks,
                    const float *a2_base, int a2_wchunks, int a2_c0, int k2chunks, int64_t rows,
                    float *out_base, int out_wchunks, int relu, int mode, psg_stream_t stream);
/* dgrad: dx = (dy W) [. (mask > 0) if mask_base]; dy is grad w.r.t. the pre-activation */
int psg_mlp_backward(const psg_mlp *m, const float *dy_base, int dy_wchunks, int64_t rows, float *dx_base,
                     int dx_wchunks, const float *mask_base, int mask_wchunks, int mode, psg_stream_t stream);

/* ---- training step of the same network (SURVEY.md 8f rank 3; train_semseg.py:164-179) ------------
 * The forward / dgrad GEMMs, grouping, max-pool, interpolation and segmented sums above are reused; these entry
 * points add what training needs.  All reductions are deterministic (fixed partitions, ordered combination). */
/* nn.BatchNorm{1,2}d.train() + optional ReLU over the rows of z (pointnet_util.py:200-203, :317-319): batch mean /
 * biased variance -> y = relu?((z - mean) * invstd * gamma + beta); running_mean / running_var (may be null) updated in
 * place with `momentum` (variance unbiased); save_mean / save_invstd [C] feed the backward.  C % 4 == 0, and every view
 * holds the C columns: 4 * z_wchunks >= C and 4 * y_wchunks >= C (else PSG_EINVAL). */
size_t psg_bn_workspace(int C);
int psg_bn_train_forward(const float *z_base, int z_wchunks, int64_t rows, int C, const float *gamma, const float *beta,
                         float *running_mean, float *running_var, float momentum, float eps, float *y_base,
                         int y_wchunks, int relu, float *save_mean, float *save_invstd, void *workspace,
                         size_t workspace_bytes, psg_stream_t stream);
/* autograd of the same: g = dy * [y > 0] (y_base null: no ReLU); dgamma = sum g xhat, dbeta = sum g,
 * dz = (g - dbeta/n - xhat dgamma/n) gamma invstd (dz may alias dy; rows past the end are zeroed).  4 * wchunks >= C for
 * dy, z, dz and (when given) y. */
int psg_bn_train_backward(const float *dy_base, int dy_wchunks, const float *y_base, int y_wchunks, const float *z_base,
                          int z_wchunks, int64_t rows, int C, const float *gamma, const float *save_mean,
                          const float *save_invstd, float *dgamma, float *dbeta, float *dz_base, int dz_wchunks,
                          void *workspace, size_t workspace_bytes, psg_stream_t stream);
/* weight / bias gradient of a 1x1 conv: dW[cout][k1+k2] (row-major) = dz^T [A1 | A2], db[cout] = column sums of dz
 * (db may be null and is overwritten; accumulate != 0 adds to dW).  Split-K over rows, partial tiles summed in order.
 * Widths: 4 * dz_wchunks >= cout; a1_c0 + ceil(k1 / 4) <= a1_wchunks, and the same for A2 when k2 > 0; k1 % 4 == 0 when
 * k2 > 0 (else PSG_EINVAL). */
size_t psg_wgrad_workspace(int cout, int cin, int64_t rows);
int psg_conv_wgrad(const float *dz_base, int dz_wchunks, int cout, const float *a1_base, int a1_wchunks, int a1_c0, int k1,
                   const float *a2_base, int a2_wchunks, int a2_c0, int k2, int64_t rows, float *dW, float *db,
                   int accumulate, void *workspace, size_t workspace_bytes, psg_stream_t stream);
/* F.log_softmax over the class logits (pointnet2_sem_seg.py:38) -> logp [rows][ncls] row-major, and its autograd.
 * 2 <= ncls <= 16 and 4 * z_wchunks >= ncls; the autograd writes all 16 columns of dz (zeros past ncls), so
 * dz_wchunks >= 4 (else PSG_EINVAL). */
int psg_log_softmax_rows(const float *z_base, int z_wchunks, int64_t rows, int ncls, float *logp, psg_stream_t stream);
int psg_dlogits_from_dlogp(const float *z_base, int z_wchunks, const float *dlogp, int64_t rows, int ncls, float *dz_base,
                           int dz_wchunks, psg_stream_t stream);
/* get_loss = F.nll_loss(pred, target, weight) (pointnet2_sem_seg.py:43-49): loss[0] = -sum w[y] logp[y] / sum w[y];
 * wsum[0] = sum w[y] (kept for the backward); labels int64; weight [ncls] or null */
size_t psg_nll_workspace(void);
int psg_nll_loss(const float *logp, const int64_t *labels, const float *weight, int64_t rows, int ncls, float *loss,
                 float *wsum, void *workspace, size_t workspace_bytes, psg_stream_t stream);
int psg_nll_loss_backward(const int64_t *labels, const float *weight, int64_t rows, int ncls, const float *grad_out,
                          const float *wsum, float *dlogp, psg_stream_t stream);
/* x *= m * scale, both T-layout [rows][C] (nn.Dropout(0.5) forward and backward with a 0/1 keep mask, scale 2);
 * 4 * x_wchunks >= C and 4 * m_wchunks >= C */
int psg_tl_mul(float *x_base, int x_wchunks, const float *m_base, int m_wchunks, int64_t rows, int C, float scale,
               psg_stream_t stream);
/* torch.optim.Adam step over one flat buffer (train_semseg.py:125-132: betas (0.9, 0.999), eps 1e-8, L2 weight_decay
 * added to the gradient); `step` counts from 1 */
int psg_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, psg_stream_t stream);

/* ---- dense kNN graph in feature space (SURVEY.md 8f rank 4; ResGCN/gcn_lib/dense/torch_edge.py:32-59) ----
 * x [B,N,C] row-major, any C >= 1, 1 <= k <= min(N, 1024) (else PSG_EINVAL): nn_idx [B,N,k] (int64, nearest first, the
 * point itself included) = the indices torch.topk(-pairwise_distance(x), k) returns; nn_d2 (optional) the squared distances,
 * equal bit for bit to psg_pairwise_distance.  Strict (distance, index) order: exact ties by ascending index, NaN distances
 * after +inf (torch.topk ranks NaN first), so every index lies in [0, N) and appears once per row, also for NaN / inf
 * features; the top-k of one k is a prefix of the top-k of a larger k.  No workspace, no [B,N,N] matrix is formed. */
int psg_dense_knn(const float *x, int B, int N, int C, int k, int64_t *nn_idx, float *nn_d2, psg_stream_t stream);
/* pairwise_distance(x) of torch_edge.py:32-43 as the full [B,N,N] matrix (API completeness, small clouds) */
int psg_pairwise_distance(const float *x, int B, int N, int C, float *out, psg_stream_t stream);

/* ---- whole-network engine (pointnet2_sem_seg.py:22-40, pointnet2_sem_seg_msg.py:23-41) -------- */
typedef struct { int cin, cout; const float *w_host; const float *b_host; } psg_mlp_desc;
typedef struct {
    int npoint, nbranch;
    double radius[2];           /* squared in double like pointnet_util.py:102 does */
    int nsample[2];
    int nlayers[2];
    psg_mlp_desc mlp[2][3];     /* first layer's input columns ordered [features | xyz] */
} psg_sa_desc;
typedef struct { int d1, d2, nlayers; psg_mlp_desc mlp[3]; } psg_fp_desc;
typedef struct {
    int in_channels, num_classes;
    psg_sa_desc sa[4];
    psg_fp_desc fp[4];          /* fp[f]: fine level f, coarse level f+1 (reference fp1 = fp[0]) */
    psg_mlp_desc conv1, conv2;
    int mlp_mode;               /* 0 = fp32 CUDA-core GEMM (exact), 1 = tcgen05 TF32 (fused kernels), 2 = tcgen05 3xTF32 (per layer, fp32-grade) */
} psg_net_desc;

/* Networks psg_net_create accepts (it returns NULL for anything else): 3-16 input channels, 2-16 classes; per SA level
 * 1-2 branches with nsample 16 or 32, npoint >= 3 and 1-3 layers; 1-3 layers per FP level; any hidden width; branch,
 * FP and conv1 outputs multiples of 16.  psg_net_bind takes any N >= npoint of SA1 (each npoint at most the previous
 * level's).  Every accepted network runs in every mode: where a width or count rules out a fused kernel or tile
 * program, that level runs per layer (tests/test_gpu_archs.py). */
typedef struct psg_net psg_net;
psg_net *psg_net_create(const psg_net_desc *desc);
void psg_net_destroy(psg_net *net);
int psg_net_set_mlp_mode(psg_net *net, int mode);
/* B blocks of N points; geometry slots for T forward passes (T*B FPS problems batched) */
size_t psg_net_workspace(const psg_net *net, int B, int N, int T);
int psg_net_bind(psg_net *net, int B, int N, int T, void *workspace, size_t workspace_bytes);
/* x [B,C,N] with element strides (sb, sc, sn): packs features and xyz */
int psg_net_set_input(psg_net *net, const float *x, int64_t sb, int64_t sc, int64_t sn, psg_stream_t stream);
/* The packed model input of `src` (as its last psg_net_set_input / psg_net_pgd_update left it) becomes the input of
 * `net`; both bound to the same B and N.  The attack loops hand a running attack from one engine to another with it
 * (nontarget.py:31-39: `color` is the PROJECTED value that enters the next forward, adv_images the un-projected one). */
int psg_net_copy_input(psg_net *net, const psg_net *src, psg_stream_t stream);
/* starts int32 [4][T][B]: FPS start index per level / forward / block (pointnet_util.py:75 draws) */
int psg_net_geometry(psg_net *net, const int32_t *starts, int T, psg_stream_t stream);
/* Copy one resident geometry buffer of forward slot t into dst (device memory, dst_bytes large enough; enqueued on
 * stream): what 0 = FPS indices of SA level (int32 [B][S]; pointnet_util.py:84), 1 = ball-query indices of SA level /
 * branch (int32 [B][S][K]; :87-107), 2 = 3-NN indices of FP level (int32 [B][Nf][3]; :302-303, level 0 = fp1 ... 3 = fp4),
 * 3 = their inverse-distance weights (float [B][Nf][3]; :304-306), 4 = coordinates of SA level (float [B][S][3]).
 * SA levels count 1..4.  These are the indices the network forward itself consumes (parity tests read them). */
int psg_net_read_geometry(const psg_net *net, int what, int level, int branch, int t, void *dst, size_t dst_bytes,
                          psg_stream_t stream);
/* forward pass t: logp [B,N,ncls] and l4_points [B,C4,16] (either may be null) */
int psg_net_forward(psg_net *net, int t, float *logp, float *l4_points, psg_stream_t stream);
/* gradient of a cost w.r.t. the logits of the last forward:
 *   kind 0: generic upstream dlogp [B,N,ncls];
 *   kind 1: cross-entropy (softmax - onehot(label or target)) * scale   (nontarget.py:34, target.py:38)
 *   kind 2: C&W f (nontarget.py:120-128), scale = sign, kappa */
int psg_net_loss_grad(psg_net *net, int kind, const float *dlogp, const int32_t *labels, int target, float scale,
                      float kappa, float *loss_rows, psg_stream_t stream);
/* input-gradient backward of forward t; grad_x [B,C,N] (feature path; may be null) */
int psg_net_backward(psg_net *net, int t, float *grad_x, psg_stream_t stream);
/* nontarget.py:37-39 / target.py:41-43 fused: adv [B,C,N] contiguous, ori [B,nc,N], mask [B,N] or null */
int psg_net_pgd_update(psg_net *net, float *adv, const float *ori, const uint8_t *mask, int c0, int nc,
                       float alpha_signed, float eps, float lo, float hi, psg_stream_t stream);
/* whole NB / tar-NB loop (nontarget.py:28-39, target.py:31-43): geometry for `iters` forwards must
 * have been built; labels int32 [B,N] (kind-1 loss), target < 0 for the non-targeted attack. */
int psg_nb_attack(psg_net *net, float *adv, const float *ori, const uint8_t *mask, const int32_t *labels,
                  int target, int iters, int t0, float alpha, float eps, float scale, psg_stream_t stream);
/* L2-ball variants of the two calls above (torchattacks PGDL2), same arguments.  Per block b, over the moving points of
 * the field (all, or mask != 0): a = cur + alpha_signed * g / (||g||_2 + 1e-10) is written to adv (un-projected), and
 * ori + (a - ori) * min(eps / ||a - ori||_2, 1), clamped to [lo, hi], becomes the next model input.  The norms are fp32
 * square roots of double sums in a fixed order: a block's result does not depend on the other blocks of the batch.
 * PSG_EINVAL for a bad field, eps < 0 or a non-finite alpha / eps. */
int psg_net_pgd_update_l2(psg_net *net, float *adv, const float *ori, const uint8_t *mask, int c0, int nc,
                          float alpha_signed, float eps, float lo, float hi, psg_stream_t stream);
int psg_nb_attack_l2(psg_net *net, float *adv, const float *ori, const uint8_t *mask, const int32_t *labels,
                     int target, int iters, int t0, float alpha, float eps, float scale, psg_stream_t stream);
/* ---- norm-unbounded attacks: NU_attack (nontarget.py:52-106), tar_NU_attack (target.py:62-133) ----
 * All buffers are caller-owned device memory.  One psg_nu_step enqueues, with no host round trip:
 * colours = (tanh(w)+1)/2 written into the model input and `adv`; forward t; C&W f and its gradient
 * (:120-128); input-gradient backward; the k-smallest colour-distance smoothness term of block 0 and
 * its gradient (:130-135); cost[step] = f + c*smooth + c*L2 and the accuracy test (:86-96) on the
 * device; the Adam update of w (torch.optim.Adam, betas 0.9/0.999, eps 1e-8).  When the accuracy
 * test fires, status[0] latches to 1 and status[1] = step; later steps leave w / adv untouched, so
 * `adv` is the image the reference returns.  status[2] = hit count of the last evaluated step. */
typedef struct {
    float *w, *adam_m, *adam_v;   /* [B,3,N] tanh-space colours and Adam moments */
    float *adv;                   /* [B,C,N] image of the last forward (the returned tensor) */
    const float *base;            /* [B,C,N] image the colours are written into (original; all-channel
                                     clamped copy after a target.py:127-132 "bingo", Q4) */
    const float *images;          /* [B,C,N] original image (L2 and smoothness reference) */
    const uint8_t *mask;          /* [B,N] points whose colours move, or null = all */
    const int32_t *labels;        /* [B,N] */
    float *cost;                  /* [>= number of steps] cost history (target.py:95) */
    int32_t *status;              /* [4] */
    float *scratch;               /* psg_nu_scratch_floats(B, N) floats */
    /* attack field: channels [field_c0, field_c0 + field_nc) move, channel j inside the tanh-space box
     * [box_lo[j], box_hi[j]].  field_nc == 0 selects the reference's field: colours 3:6 in [0,1]
     * (nontarget.py:54).  A field that includes coordinates (c0 < 3) is an extension of the reference
     * (BASELINE.json configs[2]); w / adam_m / adam_v are then [B, field_nc, N]. */
    int field_c0, field_nc;
    float box_lo[8], box_hi[8];
} psg_nu_buffers;
size_t psg_nu_scratch_floats(int B, int N);
/* w = atanh(2 colour - 1) (:57, :111-117), Adam moments and status zeroed */
int psg_nu_init(psg_net *net, const psg_nu_buffers *buf, psg_stream_t stream);
/* target < 0: f against the labels; else against `target`.  step_size = lr / (1 - 0.9^k) and
 * bc2_sqrt = sqrt(1 - 0.999^k) for the k-th step since the optimiser was (re)created; reset_adam
 * clears the moments first (target.py:123-125).  Accuracy test: hits / acc_denom  < thr
 * (exit_above = 0) or > thr (exit_above = 1), hits counted over all or only the masked points. */
int psg_nu_step(psg_net *net, const psg_nu_buffers *buf, int t, int step, int target, int neighbour, float c,
                float kappa, float targeted_sign, float step_size, float bc2_sqrt, int reset_adam, double acc_denom,
                double thr, int exit_above, int count_masked_only, const int32_t *starts, psg_stream_t stream);
/* `starts` (device int32 [4][B], or null): when the field moves coordinates the geometry of forward
 * slot t is rebuilt from the step's image with these FPS start indices before the forward pass. */

/* Also produce d cost / d xyz through the grouping and the interpolation weights (autograd of
 * pointnet_util.py:126-132, :301-308); it is added to input channels 0:3 of the feature gradient. */
int psg_net_set_xyz_grad(psg_net *net, int on);
/* x = clamp(x, lo, hi) elementwise (target.py:132 clamps all nine channels) */
int psg_clamp(float *x, int64_t count, float lo, float hi, psg_stream_t stream);

/* Per-class counters of NB_nontarget_test_semseg.py:187-211 / NB_target_test_semseg.py:187-190 as one
 * histogram: conf is int64 [ncls*ncls + 4] and is ACCUMULATED into: conf[label*ncls + pred] += 1 with
 * pred = first arg-max of logp [rows,ncls]; then rows seen, rows with pred == label, masked rows,
 * masked rows with pred == target (mask optional).  This buffer is what the NCCL all-reduce sums. */
int psg_confusion_matrix(const float *logp, const int32_t *labels, const uint8_t *mask, int target, int64_t rows,
                         int ncls, int64_t *conf, psg_stream_t stream);
/* Whole-scene voting, add_vote of NB_nontarget_test_semseg.py:55-62 (SURVEY.md 8f rank 1): for every row with
 * weight != 0 (weight may be null = all), pool[point_idx[row]][first arg-max of logp[row]] += 1.  pool is
 * float32 [pool_rows][ncls] holding exact integer counts; psg_confusion_matrix(pool, scene_labels, ...)
 * then yields the scene-level seen / correct / union counters of :216-241 (np.argmax = first arg-max),
 * and under sharding the pool is what ranks all-reduce. */
int psg_add_vote(const float *logp, const int64_t *point_idx, const float *weight, int64_t rows, int ncls, float *pool,
                 int64_t pool_rows, psg_stream_t stream);

/* ---- whole-scene block slicer (SURVEY.md 8f rank 2): ScannetDatasetWholeScene.__getitem__,
 * data_utils/S3DISDataLoader.py:124-175.  `points` is the room, float64 [P][ld] row-major with x, y, z, r, g, b in
 * columns 0..5 and the label in column label_col; it stays resident on the device.  Columns ("cells") are the
 * reference's grid_y x grid_x loop in row-major order; their padded bounds (lo_x, hi_x, lo_y, hi_y), their centres
 * (s_x + block_size / 2, s_y + block_size / 2) and the random positions are computed by the host mirror
 * (pointsecguard_b200/data_utils/S3DISDataLoader.py) with the reference's float64 expressions and numpy draws. ---- */

/* room bounding box, :128: out6 = (min x, y, z, max x, y, z).  The workspace must be zero-filled once by the caller. */
size_t psg_scene_minmax_workspace(void);
int psg_scene_minmax(const double *points, int64_t P, int ld, double *out6, void *workspace, size_t workspace_bytes,
                     psg_stream_t stream);
/* number of 1024-point chunks the passes below split P points into */
int64_t psg_scene_chunks(int64_t P);
/* np.where of :143-145, pass 1: counts [ncell][chunks] receives, per column, the EXCLUSIVE scan over chunks of its
 * member counts; totals [ncell] the members per column (= point_idxs.size of :146, what the host's draws depend on) */
int psg_scene_cell_counts(const double *points, int64_t P, int ld, const double *cell_bounds, int ncell, int32_t *counts,
                          int32_t *totals, psg_stream_t stream);
/* pass 2: sel[cell_offset[c] + k] = k-th smallest member index of column c (cell_offset = exclusive sum of totals) */
int psg_scene_cell_fill(const double *points, int64_t P, int ld, const double *cell_bounds, int ncell,
                        const int32_t *counts, const int64_t *cell_offset, int32_t *sel, psg_stream_t stream);
/* :155-166 for all blocks at once.  Output row r belongs to block r / block_points of column block_cell[block] and
 * takes member number row_pos[r] of that column (the host's choice + shuffle).  data [rows][9] float64 (optional),
 * data32 the same rounded to float32 as torch.Tensor(ndarray) does (optional), label int64, smpw float64 =
 * labelweights[label], index int64 = the point's row in the room (each optional). */
int psg_scene_gather(const double *points, int ld, int label_col, const int32_t *sel, const int64_t *cell_offset,
                     const int32_t *block_cell, const int32_t *row_pos, const double *centre, const double *room_max,
                     const float *labelweights, int ncls, int64_t rows, int block_points, double *data, float *data32,
                     int64_t *label, double *smpw, int64_t *index, psg_stream_t stream);

/* library-wide switches; unknown names return PSG_EINVAL.
 * "nn_grid" (default 0) = 3-NN search over a grid of the coarse cloud: 0 automatic, 1 never, 2 whenever it fits;
 * "fps_cluster" (default 1) = cluster FPS kernel for large clouds;
 * "sa_compact" (default 1) = fused set-abstraction branches run on compacted neighbourhood rows (0: padded rows);
 * "x3_fused" (default 3) = 3xTF32 mode: bit 0 fuses the narrow set-abstraction branches, bit 1 fp1 + head;
 * "stream_stages", "stream_stage_bytes", "stream_rings" = ring of psg_debug_l2_stream (measurement only) */
int psg_set_option(const char *name, int value);
/* Measurement only (tools/l2_stream_bench.py): `ctas` CTAs each stream `passes` x region_bytes of L2-resident memory into
 * shared memory with bulk async copies.  mode 0: CTA (or cluster) i reads region i of buf; mode 1: all read region 0.
 * cluster in {1, 2, 4, 8}: the CTAs of a cluster want the same bytes and fetch them once, by multicast. */
int psg_debug_l2_stream(const void *buf, int64_t region_bytes, int mode, int cluster, int passes, int ctas, psg_stream_t stream);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
int64_t psg_launch_count(void);
/* per-kernel-family device timing of the engine (CUDA event pairs on the launching stream);
 * collect() synchronises the device, fills ms / launch counts per family and resets. */
int psg_prof_enable(int on);
int psg_prof_ncat(void);
const char *psg_prof_name(int cat);
int psg_prof_collect(double *ms_by_cat, int64_t *count_by_cat);
/* debug: CTA 0 of each of the next `nlaunches` tile-program launches (csrc/chain_fused.cu) writes clock64
 * stamps of its phases into buf ([nlaunches][4 roles][512] int64: worker tile 0, worker tile 1, MMA issuer);
 * buf = NULL switches it off -- tools/tile_trace.py */
int psg_debug_trace(int64_t *buf, int nlaunches);

#ifdef __cplusplus
}
#endif
#endif
