// psg_internal.h -- launcher prototypes shared by the translation units of libpsg_b200.
// Nothing here is part of the C ABI (see include/psg_b200.h for that).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "psg_common.cuh"

enum { PSG_EPI_BIAS_RELU = 0, PSG_EPI_BIAS = 1, PSG_EPI_MASK = 2, PSG_EPI_NONE = 3 };

struct PsgGemmArgs {
    TView A1; int k1chunks;     // first K1 = 4*k1chunks columns of the A operand
    TView A2; int k2chunks;     // optional second source (FP concat); k2chunks = 0 if unused
    const float *W; int Nw;     // packed weights [K/4][Nw][4], Nw = output channels padded to 64
    const float *Wlo;           // tcgen05 path: W is W_hi and this the TF32 residual W_lo (error-compensated 3xTF32), or null
    const float *bias;          // [nout_pad] (zero padded) or null
    TView Out; int nout_pad;    // columns written (multiple of 16)
    TView Mask;                 // PSG_EPI_MASK: forward activation of the layer below
    int mtiles;                 // padded rows / 128
    int epi;
    TView Out2; int out2_cols;  // optional: columns [0, out2_cols) are ALSO written here (tcgen05 path; FP skip-gradient)
};

// slicer.cu (whole-scene block slicer, SURVEY.md 8f rank 2)
size_t psg_scene_minmax_ws_bytes();
int psg_scene_minmax_k(const double *pts, long long P, int ld, double *out6, void *ws, cudaStream_t st);
int psg_scene_count_k(const double *pts, long long P, int ld, const double *bounds, int ncell, int *counts, int *totals,
                      cudaStream_t st);
int psg_scene_fill_k(const double *pts, long long P, int ld, const double *bounds, int ncell, const int *counts,
                     const long long *cell_off, int *sel, cudaStream_t st);
int psg_scene_gather_k(const double *pts, int ld, int label_col, const int *sel, const long long *cell_off, const int *block_cell,
                       const int *row_pos, const double *centre, const double *room_max, const float *labelweights, int ncls,
                       long long rows, int block_points, double *data, float *data32, long long *label, double *smpw,
                       long long *index, cudaStream_t st);

// fps.cu
void psg_fps_use_cluster(int on);
size_t psg_fps_workspace_bytes(int P, int N);
int psg_fps_launch(const float *xyz, long long cloud_stride, int nclouds, int P, int N, int npoint,
                   const int *start, int *out_idx, float *out_xyz, void *ws, size_t ws_bytes, cudaStream_t st);
// neighbors.cu
int psg_ball_query_launch(const float *xyz, long long cloud_stride, int nclouds, int P, int N,
                          const float *new_xyz, int S, int nr, const double *radius, const int *nsample,
                          int *out0, int *out1, cudaStream_t st);
int psg_three_nn_launch(const float *xyz1, long long stride1, int nclouds1, int P, int N,
                        const float *xyz2, int S, int *idx, float *w, float *d2, cudaStream_t st);
void psg_three_nn_grid_mode(int m);   // 0 automatic, 1 never, 2 always (A/B and tests)
int psg_square_distance_launch(const float *src, const float *dst, int B, int N, int M, float *out, cudaStream_t st);
// ballgrid.cu: ball query over a uniform grid (large clouds), same results as psg_ball_query_launch
size_t psg_ballgrid_workspace_bytes(int nclouds, int N);
int psg_ballgrid_build(const float *xyz, long long cloud_stride, int nclouds, int N, double rmax, void *ws, cudaStream_t st);
int psg_ballgrid_query(const void *ws, const float *xyz, long long cloud_stride, int nclouds, int P, int N, const float *new_xyz,
                       int S, int nr, const double *radius, const int *nsample, int *out0, int *out1, cudaStream_t st);
// gather.cu
int psg_pack_cf(const float *x, long long sb, long long sc, long long sn, int B, int C, int N, TView out,
                int cpad, float *xyz, cudaStream_t st);
int psg_unpack_cf(TView in, int B, int C, int N, float *y, int accumulate, cudaStream_t st);
int psg_pack_rm(const float *x, long long rows, int C, TView out, int cpad, cudaStream_t st);
int psg_unpack_rm(TView in, long long rows, int C, float *y, cudaStream_t st);
int psg_group(TView feats, int D, const float *xyz, long long cloud_stride, int nclouds, int Nsrc,
              const float *new_xyz, const int *idx, int P, int S, int K, TView out, int cpad, cudaStream_t st);
int psg_maxpool(TView in, long long groups, int K, int C, TView out, unsigned char *arg, cudaStream_t st);
int psg_maxpool_bwd(TView dout, TView outv, const unsigned char *arg, long long groups, int K, int C, TView dy,
                    cudaStream_t st);
int psg_interp(TView feats, int S, const int *idx, const float *w, long long P, int N, int nch, TView out,
               cudaStream_t st);
size_t psg_csr_scratch_bytes(long long P, int M, int R);
int psg_csr_build(const int *keys, long long P, int M, int R, int grp, int *offs, int *perm, void *scratch, cudaStream_t st);
int psg_segsum(TView src, long long src_rows_per_p, int div, const float *wgt, const int *offs, const int *perm,
               int M, int R, long long P, int ncols, TView dst, int accumulate, const TView *relu_mask, const float *src_rm,
               int rm_stride, cudaStream_t st);
int psg_copy_cols(TView src, TView dst, long long rows, int ncols, int accumulate, cudaStream_t st);
int psg_index_points_rm(const float *pts, const long long *idx, int B, int N, int C, long long M, float *out,
                        cudaStream_t st);
// train.cu
int psg_repack_weights(const float *w, const float *b, int cout, int cin, int kpad, int npad, int nwf, int nwb, float *wf,
                       float *wb, float *wf_c, float *wb_c, float *bias, float comp, cudaStream_t st);
// streambench.cu (measurement only)
void psg_stream_tune(int stages, int stage_bytes, int rings);
// gemm_simt.cu / gemm_tc.cu
int psg_gemm_simt(const PsgGemmArgs &g, cudaStream_t st);
int psg_gemm_tc(const PsgGemmArgs &g, cudaStream_t st);
// sa_fused.cu: one set-abstraction branch (gather -> 3 layers -> neighbourhood max) per kernel
// compact.cu: compacted neighbourhood rows (real ball-query hits only) of one fused SA branch
struct PsgCompact {
    int *cnt;        // [P*S] real hits of each neighbourhood
    int *slot;       // [P*S] octet position of the neighbourhood inside its problem's compact rows
    int *nsl;        // [P]   32-row slices used by the problem
    int *base;       // [P]   first compact row of the problem inside its forward's row space
    int *ctiles;     // [T]   128-row tiles of each forward
    int *crow_src;   // [T][B*S*K] source point of each compact row (-1: empty)
    int *crow_g;     // [T][B*S*K] centroid (b*S + s) of each compact row (-1: empty)
    int *cperm;      // [P][S*K] gather-backward CSR permutation rewritten to compact rows (relative to the forward)
    long long cap;
};
size_t psg_sa_compact_bytes(long long P, int T, int S, int K);
PsgCompact psg_sa_compact_carve(void *ws, long long P, int T, int S, int K);
int psg_sa_compact_build(const int *ball, const int *csr_perm, int T, int B, int S, int K, PsgCompact c, cudaStream_t st);
bool psg_sa_compactable(int K, int gpad, int n0, int n1, int n2);

struct PsgSaFused {
    int K;
    TView feats; int D; const float *xyz; long long cloud_stride; int nclouds; int Nsrc;
    const float *new_xyz; const int *idx; long long rows; int S;
    int gpad; int n[3];
    const float *wf[3]; int nwf[3]; const float *bias[3];
    const float *wb[3]; int nwb[3];
    unsigned *m0, *m1;             // ReLU bits of layers 0 / 1, psg_sa_mask_words(rows, n) words each
    TView out; unsigned char *arg; // pooled rows [groups][n2 slice of the level's features], arg-max [groups][n2]
    // compacted rows (compact.cu), all null for the padded [S][K] layout: per compact row its source point / centroid, and
    // the forward's tile count in device memory (only the device knows how many real hits there are)
    const int *crow_src, *crow_g, *ntiles_dev;
    // 3xTF32 (mode 2): TF32 residuals of wf / wb in the same packings (wf / wb are then the "hi" parts); all null otherwise
    const float *wf_lo[3], *wb_lo[3];
};
bool psg_sa_fusable(int K, int gpad, int n0, int n1, int n2);
bool psg_sa_fusable_x3(int K, int gpad, int n0, int n1, int n2);
size_t psg_sa_mask_words(long long rows, int n);
int psg_sa_fused_fwd(const PsgSaFused &f, cudaStream_t st);
int psg_sa_fused_bwd(const PsgSaFused &f, TView dout, TView dG, int gcols, float *dG_rm, int rm_only, cudaStream_t st);
// chain_fused.cu: finest FP level + head, forward [+ loss gradient + backward] in one kernel
#define PSG_CHAIN_MAX_OPS 10
struct PsgChain {
    TView src; int S; const int *nn_idx; const float *nn_w; int Nf; int kin; long long rows;
    const float *src_rm;               // row-major mirror of src ([rows of src][kin]) or null
    int nlayers;                       // hidden layers (conv + folded BN + ReLU), <= 4
    int n[4]; const float *wf[4]; int nwf[4]; const float *bias[4]; const float *wb[4]; int nwb[4];
    const float *head_wf; int head_nwf; const float *head_bias; const float *head_wb; int head_nwb;
    int backward;                      // 0: logits -> zout; 1: loss gradient + dgrad chain -> dI
    int ncls, loss_kind, target; const int *labels; float scale, kappa; const float *dlogp;
    float *loss_rows; unsigned char *hit;
    TView zout, dI;
    float *dI_rm; int rm_only;         // row-major copy of dI ([rows][kin]) for the segmented sum; rm_only: skip the T-layout store
    // 3xTF32 (mode 2): the TF32 residuals of every weight above (wf / wb / head_* are then the "hi" parts); all null otherwise
    const float *wf_lo[4], *wb_lo[4], *head_wf_lo, *head_wb_lo;
};
int psg_chain_fused(const PsgChain &c, cudaStream_t st);
// set-abstraction branch with streamed weights (widths beyond what sa_fused.cu keeps resident)
bool psg_sa_streamable(int K, int gpad, int n0, int n1, int n2);
int psg_sa_stream_fwd(const PsgSaFused &f, cudaStream_t st);
int psg_sa_stream_bwd(const PsgSaFused &f, TView dout, TView dG, int gcols, float *dG_rm, int rm_only, cudaStream_t st);
// feature-propagation level: [skip | 3-NN interpolation] -> MLP, forward and dgrad chain
struct PsgFpStream {
    TView skip; int C1; TView coarse; int C2, S, Nf; const int *nn_idx; const float *nn_w; long long rows;
    int nl; int n[3]; const float *wf[3]; int nwf[3]; const float *bias[3]; const float *wb[3]; int nwb[3];
    unsigned *m[3];                    // ReLU bits of the hidden layers
    TView y_last;                      // output of the last layer (stored: next level's interpolation source)
    float *y_last_rm;                  // optional row-major mirror of y_last ([rows][n_last]) for the next level's gather
    const float *coarse_rm;            // optional row-major mirror of `coarse` ([rows][C2])
};
bool psg_fp_streamable(const PsgFpStream &f, bool forward);
int psg_fp_stream_fwd(const PsgFpStream &f, cudaStream_t st);
// psg_fp_stream_bwd also writes the first psg_fp_stream_skip_cols(f) columns of d[skip] into dskip; the caller copies
// the remaining C1 - psg_fp_stream_skip_cols(f) columns out of dcat
int psg_fp_stream_bwd(const PsgFpStream &f, TView dy_last, TView dcat, float *dcat_rm, TView dskip, cudaStream_t st);
int psg_fp_stream_skip_cols(const PsgFpStream &f);
long long *psg_tile_trace_slot();   // next [4][512] block of the debug trace buffer, or null
void psg_tile_set_trace(long long *buf, int nlaunches);
// geomgrad.cu: gradient w.r.t. coordinates through grouping and interpolation weights
int psg_sa_xyz_backward(TView dG, int D, int K, long long groups_per_p, long long P, const int *offs, const int *perm, int R,
                        float *dxyz_src, float *dxyz_ctr, cudaStream_t st);
int psg_fps_xyz_backward(const float *dxyz_l, const int *fps_idx, int S, int R, int P, float *dxyz_src, cudaStream_t st);
int psg_fp_xyz_backward(TView dI, TView coarse, int C2, const float *xyz1, long long stride1, int nclouds1, const float *xyz2,
                        int S, const int *nn_idx, const int *offs, const int *perm, long long P, int N, float *dxyz1,
                        float *dxyz2, float *ctmp, cudaStream_t st);
int psg_add_xyz_to_feat(const float *dxyz0, long long rows, TView dfeat0, cudaStream_t st);
// elementwise.cu
int psg_head_logsoftmax(TView z, long long rows, int ncls, float *logp, cudaStream_t st);
int psg_dz_from_dlogp(TView z, const float *dlogp, long long rows, int ncls, TView dz, cudaStream_t st);
int psg_dz_ce(TView z, const int *labels, int target, long long rows, int ncls, float scale, TView dz,
              cudaStream_t st);
int psg_dz_cw(TView z, const int *labels, int target, long long rows, int ncls, float kappa, float sign, TView dz,
              float *loss_rows, unsigned char *hit, cudaStream_t st);
int psg_pgd_update(float *adv, const float *ori, TView grad, TView feats0, const unsigned char *mask, int B, int C,
                   int N, int c0, int nc, float alpha_signed, float eps, float lo, float hi, cudaStream_t st);
int psg_pgd_l2_update(float *adv, const float *ori, TView grad, TView feats0, const unsigned char *mask, int B, int C,
                      int N, int c0, int nc, float alpha_signed, float eps, float lo, float hi, cudaStream_t st);
int psg_confusion(const float *logp, const int *labels, const unsigned char *mask, int target, long long rows, int ncls,
                  long long *conf, cudaStream_t st);
int psg_add_vote_k(const float *logp, const long long *point_idx, const float *weight, long long rows, int ncls, float *pool,
                   long long pool_rows, cudaStream_t st);
// nu.cu
struct PsgNuField { int c0, nc; float lo[8], hi[8]; };   // perturbed channels [c0, c0+nc) and their tanh-space box
int psg_nu_init_k(const float *images, int B, int C, int N, PsgNuField fld, float *w, float *m, float *v, cudaStream_t st);
int psg_nu_build_adv_k(const float *w, const float *base, const float *images, const unsigned char *mask, int B, int C,
                     int N, PsgNuField fld, TView feats0, float *adv, float *l2_rows, const int *status, cudaStream_t st);
int psg_nu_smooth_k(const float *adv0, const float *images0, int C, int N, int k, float *rows_out, float *grad_out,
                  cudaStream_t st);
int psg_nu_reduce_k(const float *f_rows, const float *l2_rows, const float *smooth_rows, const unsigned char *hit,
                  const unsigned char *mask, long long rows, int nsmooth, float c, int step, double acc_denom, double thr,
                  int exit_above, int count_masked_only, float *cost, int *status, cudaStream_t st);
int psg_nu_adam_k(float *w, float *m, float *v, TView grad0, const float *adv, const float *images,
                const float *smooth_grad, const unsigned char *mask, int B, int C, int N, PsgNuField fld, float c, float step_size,
                float bc2_sqrt, float beta1, float beta2, float eps, int reset, const int *status, cudaStream_t st);
int psg_clamp_k(float *x, long long n, float lo, float hi, cudaStream_t st);
