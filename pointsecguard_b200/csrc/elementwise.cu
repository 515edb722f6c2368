// elementwise.cu -- head, loss gradients, the fused perturbation update and the metric histogram.
// Reference: pointnet2_sem_seg.py:36-39 (log_softmax head), nontarget.py:26,34 / target.py:27,38
// (cross-entropy costs), nontarget.py:120-128 (C&W f), nontarget.py:37-39 / target.py:41-43 (PGD
// update + projection), NB_nontarget_test_semseg.py:187-211 (per-class counters).
#include "psg_common.cuh"
#include "psg_internal.h"
#include "psg_loss.cuh"

namespace {

constexpr int kMaxCls = 16;

__device__ __forceinline__ void load_row(const TView &z, long long row, int ncls, float *v)
{
#pragma unroll
    for (int c = 0; c < kMaxCls / 4; ++c) {
        if (4 * c < ncls) {
            float4 q = tv_ld(z, row, c);
            v[4 * c] = q.x; v[4 * c + 1] = q.y; v[4 * c + 2] = q.z; v[4 * c + 3] = q.w;
        }
    }
}
__device__ __forceinline__ void store_row(const TView &z, long long row, const float *v)
{
#pragma unroll
    for (int c = 0; c < kMaxCls / 4; ++c) tv_st(z, row, c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
}
__device__ __forceinline__ void softmax_row(const float *v, int ncls, float *p, float &mx, float &lse)
{
    psg_softmax_row(v, ncls, p, mx, lse);
}

__global__ void head_logsoftmax_kernel(TView z, long long rows, int ncls, float *__restrict__ logp)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float v[kMaxCls], p[kMaxCls], mx, lse;
    load_row(z, row, ncls, v);
    softmax_row(v, ncls, p, mx, lse);
    for (int c = 0; c < ncls; ++c) logp[row * ncls + c] = (v[c] - mx) - lse;
}

// generic upstream gradient on the log-probabilities: dz = dlogp - softmax * sum(dlogp)
__global__ void dz_from_dlogp_kernel(TView z, const float *__restrict__ dlogp, long long rows, int ncls, TView dz)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float v[kMaxCls], o[kMaxCls];
    load_row(z, row, ncls, v);
    psg_dz_generic(v, ncls, dlogp + row * ncls, o);
    store_row(dz, row, o);
}

__global__ void dz_ce_kernel(TView z, const int *__restrict__ labels, int target, long long rows, int ncls,
                             float scale, TView dz)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float v[kMaxCls], o[kMaxCls];
    load_row(z, row, ncls, v);
    psg_dz_ce_row(v, ncls, target >= 0 ? target : labels[row], scale, o);
    store_row(dz, row, o);
}

__global__ void dz_cw_kernel(TView z, const int *__restrict__ labels, int target, long long rows, int ncls,
                             float kappa, float sgn, TView dz, float *__restrict__ loss_rows,
                             unsigned char *__restrict__ hit)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float v[kMaxCls], o[kMaxCls];
    load_row(z, row, ncls, v);
    int h;
    const float f = psg_dz_cw_row(v, ncls, target >= 0 ? target : labels[row], kappa, sgn, o, h);
    if (loss_rows) loss_rows[row] = f;
    if (hit) hit[row] = (unsigned char)h;
    store_row(dz, row, o);
}

// One step of nontarget.py:37-39 / target.py:41-43 on channels [c0, c0+nc):
//   a   = cur + alpha_signed * sign(g)         -> adv (the reference returns this un-projected value)
//   eta = clamp(a - ori, +-eps); col = clamp(ori + eta, lo, hi) -> next model input (feats0)
__global__ void pgd_update_kernel(float *__restrict__ adv, const float *__restrict__ ori, TView grad, TView feats0,
                                  const unsigned char *__restrict__ mask, int B, int C, int N, int c0, int nc,
                                  float alpha_signed, float eps, float lo, float hi)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");          // launched with programmatic stream serialization
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= (long long)B * N) return;
    const int b = (int)(row / N), n = (int)(row % N);
    // target.py:41-43 reads and writes the masked points only: everything else keeps its input value, unclamped
    if (mask && mask[row] == 0) return;
    for (int j = 0; j < nc; ++j) {
        const int ch = c0 + j;
        float *fp = feats0.base + tv_off(feats0, row, ch >> 2) + (ch & 3);
        const float cur = *fp;
        const float g = grad.base[tv_off(grad, row, ch >> 2) + (ch & 3)];
        const float sg = g > 0.f ? 1.f : (g < 0.f ? -1.f : 0.f);
        const float a = __fadd_rn(cur, __fmul_rn(alpha_signed, sg));
        const float o = ori[((long long)b * nc + j) * N + n];
        adv[((long long)b * C + ch) * N + n] = a;
        const float eta = fminf(fmaxf(__fsub_rn(a, o), -eps), eps);
        *fp = fminf(fmaxf(__fadd_rn(o, eta), lo), hi);
    }
}

// L2-ball variant of the step above (torchattacks PGDL2), one CTA per block b over its moving points (all, or the masked):
//   gn = fp32(sqrt(sum double(g)^2));  a = cur + alpha_signed * (g / (gn + 1e-10f))  -> adv (un-projected, as above)
//   d = a - ori;  dn = fp32(sqrt(sum double(d)^2));  f = dn > eps ? eps / dn : 1;  col = clamp(ori + d * f, lo, hi) -> feats0
// Every element op is separately rounded fp32.  The sums are per-thread partials in a fixed point order, a fixed shuffle
// tree and a warp-order pass, so a block's result depends on N and its own data only (not on B, sharding or chunking).
constexpr int kL2Threads = 512;

__device__ __forceinline__ double l2_block_sum(double v, double *sh)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kL2Threads / 32; ++w) s = __dadd_rn(s, sh[w]);
    __syncthreads();                                               // sh is reused by the next sum
    return s;
}

__global__ void __launch_bounds__(kL2Threads) pgd_l2_update_kernel(float *__restrict__ adv, const float *__restrict__ ori,
                                                                  TView grad, TView feats0,
                                                                  const unsigned char *__restrict__ mask, int C, int N,
                                                                  int c0, int nc, float alpha_signed, float eps, float lo,
                                                                  float hi)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");          // launched with programmatic stream serialization
    __shared__ double sh[kL2Threads / 32];
    const int b = blockIdx.x;
    const long long row0 = (long long)b * N;
    const unsigned char *mk = mask ? mask + row0 : nullptr;
    auto g_at = [&](int n, int ch) { return grad.base[tv_off(grad, row0 + n, ch >> 2) + (ch & 3)]; };
    auto f_at = [&](int n, int ch) { return feats0.base + tv_off(feats0, row0 + n, ch >> 2) + (ch & 3); };

    double s = 0.0;                                                // pass 1: sum g^2
    for (int n = threadIdx.x; n < N; n += kL2Threads) {
        if (mk && mk[n] == 0) continue;
        for (int j = 0; j < nc; ++j) {
            const double g = g_at(n, c0 + j);
            s = __dadd_rn(s, __dmul_rn(g, g));
        }
    }
    const float den = __fadd_rn(__double2float_rn(sqrt(l2_block_sum(s, sh))), 1e-10f);

    s = 0.0;                                                       // pass 2: write adv, sum d^2
    for (int n = threadIdx.x; n < N; n += kL2Threads) {
        if (mk && mk[n] == 0) continue;
        for (int j = 0; j < nc; ++j) {
            const int ch = c0 + j;
            const float a = __fadd_rn(*f_at(n, ch), __fmul_rn(alpha_signed, __fdiv_rn(g_at(n, ch), den)));
            adv[((long long)b * C + ch) * N + n] = a;
            const double d = __fsub_rn(a, ori[((long long)b * nc + j) * N + n]);
            s = __dadd_rn(s, __dmul_rn(d, d));
        }
    }
    const float dn = __double2float_rn(sqrt(l2_block_sum(s, sh)));
    const float f = dn > eps ? __fdiv_rn(eps, dn) : 1.f;

    for (int n = threadIdx.x; n < N; n += kL2Threads) {            // pass 3: the same a and d, projected and clamped
        if (mk && mk[n] == 0) continue;
        for (int j = 0; j < nc; ++j) {
            const int ch = c0 + j;
            float *fp = f_at(n, ch);
            const float a = __fadd_rn(*fp, __fmul_rn(alpha_signed, __fdiv_rn(g_at(n, ch), den)));
            const float o = ori[((long long)b * nc + j) * N + n];
            *fp = fminf(fmaxf(__fadd_rn(o, __fmul_rn(__fsub_rn(a, o), f)), lo), hi);
        }
    }
}

// conf[label][pred] += 1 with pred = first arg-max of the log-probabilities, followed by four
// scalars: rows seen, rows with pred == label, masked rows, masked rows with pred == target
__global__ void confusion_kernel(const float *__restrict__ logp, const int *__restrict__ labels,
                                 const unsigned char *__restrict__ mask, int target, long long rows,
                                 int ncls, unsigned long long *__restrict__ conf)
{
    __shared__ unsigned int h[kMaxCls * kMaxCls + 4];
    const int nh = ncls * ncls + 4;
    for (int i = threadIdx.x; i < nh; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x; row < rows;
         row += (long long)gridDim.x * blockDim.x) {
        const float *v = logp + row * ncls;
        int best = 0; float bv = v[0];
        for (int c = 1; c < ncls; ++c) if (v[c] > bv) { bv = v[c]; best = c; }
        const int y = labels[row];
        if (y >= 0 && y < ncls) atomicAdd(&h[y * ncls + best], 1u);
        atomicAdd(&h[ncls * ncls], 1u);
        if (best == y) atomicAdd(&h[ncls * ncls + 1], 1u);
        if (mask && mask[row]) {
            atomicAdd(&h[ncls * ncls + 2], 1u);
            if (best == target) atomicAdd(&h[ncls * ncls + 3], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nh; i += blockDim.x)
        if (h[i]) atomicAdd(conf + i, (unsigned long long)h[i]);
}

// add_vote of the attack scripts (NB_nontarget_test_semseg.py:55-62): for every block point with a
// non-zero weight, vote_label_pool[point_idx, argmax(logp)] += 1.  The pool holds small exact integers
// in float32, so the atomic adds commute exactly and the result is run-to-run identical.
__global__ void add_vote_kernel(const float *__restrict__ logp, const long long *__restrict__ point_idx,
                                const float *__restrict__ weight, long long rows, int ncls, float *__restrict__ pool,
                                long long pool_rows)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    if (weight && weight[row] == 0.f) return;
    const long long pi = point_idx[row];
    if (pi < 0 || pi >= pool_rows) return;
    const float *v = logp + row * ncls;
    int best = 0; float bv = v[0];
    for (int c = 1; c < ncls; ++c) if (v[c] > bv) { bv = v[c]; best = c; }
    atomicAdd(pool + pi * ncls + best, 1.0f);
}

inline unsigned nb(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

int psg_head_logsoftmax(TView z, long long rows, int ncls, float *logp, cudaStream_t st)
{
    if (ncls > kMaxCls) return PSG_EUNSUPPORTED;
    head_logsoftmax_kernel<<<nb(rows, 256), 256, 0, st>>>(z, rows, ncls, logp);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_dz_from_dlogp(TView z, const float *dlogp, long long rows, int ncls, TView dz, cudaStream_t st)
{
    if (ncls > kMaxCls) return PSG_EUNSUPPORTED;
    dz_from_dlogp_kernel<<<nb(rows, 256), 256, 0, st>>>(z, dlogp, rows, ncls, dz);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_dz_ce(TView z, const int *labels, int target, long long rows, int ncls, float scale, TView dz, cudaStream_t st)
{
    if (ncls > kMaxCls) return PSG_EUNSUPPORTED;
    dz_ce_kernel<<<nb(rows, 256), 256, 0, st>>>(z, labels, target, rows, ncls, scale, dz);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_dz_cw(TView z, const int *labels, int target, long long rows, int ncls, float kappa, float sign, TView dz,
              float *loss_rows, unsigned char *hit, cudaStream_t st)
{
    if (ncls > kMaxCls) return PSG_EUNSUPPORTED;
    dz_cw_kernel<<<nb(rows, 256), 256, 0, st>>>(z, labels, target, rows, ncls, kappa, sign, dz, loss_rows, hit);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_pgd_update(float *adv, const float *ori, TView grad, TView feats0, const unsigned char *mask, int B, int C,
                   int N, int c0, int nc, float alpha_signed, float eps, float lo, float hi, cudaStream_t st)
{
    if (psg_launch_pdl(pgd_update_kernel, dim3(nb((long long)B * N, 256)), dim3(256), 0, st, 1, adv, ori, grad, feats0, mask, B, C, N, c0,
                       nc, alpha_signed, eps, lo, hi) != cudaSuccess) return PSG_ECUDA;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_pgd_l2_update(float *adv, const float *ori, TView grad, TView feats0, const unsigned char *mask, int B, int C,
                      int N, int c0, int nc, float alpha_signed, float eps, float lo, float hi, cudaStream_t st)
{
    if (psg_launch_pdl(pgd_l2_update_kernel, dim3((unsigned)B), dim3(kL2Threads), 0, st, 1, adv, ori, grad, feats0, mask, C,
                       N, c0, nc, alpha_signed, eps, lo, hi) != cudaSuccess) return PSG_ECUDA;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_confusion(const float *logp, const int *labels, const unsigned char *mask, int target, long long rows, int ncls,
                  long long *conf, cudaStream_t st)
{
    if (ncls > kMaxCls) return PSG_EUNSUPPORTED;
    const unsigned blocks = (unsigned)min((long long)592, (rows + 255) / 256);
    confusion_kernel<<<blocks, 256, 0, st>>>(logp, labels, mask, target, rows, ncls, (unsigned long long *)conf);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

int psg_add_vote_k(const float *logp, const long long *point_idx, const float *weight, long long rows, int ncls, float *pool,
                   long long pool_rows, cudaStream_t st)
{
    add_vote_kernel<<<nb(rows, 256), 256, 0, st>>>(logp, point_idx, weight, rows, ncls, pool, pool_rows);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
