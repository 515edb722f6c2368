// train.cu -- kernels of the TRAINING step of the same network (SURVEY.md 8f rank 3).
//
// Reference: PointNet/train_semseg.py:164-179 (classifier.train(); forward; get_loss; loss.backward(); optimizer.step()),
// nn.BatchNorm{1,2}d in train mode inside PointNet/models/pointnet_util.py:200-203, :256-260, :317-319 and
// pointnet2_sem_seg.py:35, F.nll_loss with class weights (pointnet2_sem_seg.py:47), torch.optim.Adam with L2 weight decay
// (train_semseg.py:125-132).
//
// What training adds to the attack path's kernels (gather, grouping, max-pool, interpolation, dgrad GEMMs, segmented
// sums -- all reused): batch statistics and their backward, weight / bias gradients, the weighted NLL, Adam.
// Everything is deterministic: column reductions run over a fixed row partition with double-precision partial sums that
// are combined in order; wgrad is a split-K GEMM whose partial tiles are summed in split order.  All activations are
// T-layout (psg_common.cuh).
#include "../../include/psg_b200.h"
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

inline TView mkv(const float *base, int wchunks, int c0) { return TView{const_cast<float *>(base), wchunks, c0}; }

// ------------------------------------------------------------------------------------------------
// column reductions over the rows of a T-layout tensor: grid (chunks, splits), 256 threads, thread = one row of a
// 128-row tile (two tiles per pass), four channels per thread.  MODE 0: sum z, sum z^2 (batch statistics);
// MODE 1: sum g, sum g * xhat with g = dy * [y > 0] (BatchNorm backward); MODE 2: sum z only (bias gradient).
// ------------------------------------------------------------------------------------------------
struct ColRedArgs {
    TView a, b, c;              // MODE 0/2: a = z;  MODE 1: a = dy, b = y (ReLU mask, may be null), c = z
    const float *mean, *invstd; // MODE 1
    long long rows;
    int ntiles, tiles_per_split;
    double *partial;            // [splits][C][2]
    int C;
};

template <int MODE>
__global__ void __launch_bounds__(256) colred_kernel(ColRedArgs p)
{
    const int chunk = blockIdx.x, split = blockIdx.y;
    const int r = threadIdx.x & 127, half = threadIdx.x >> 7;
    double s[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
    float mu[4] = {0, 0, 0, 0}, is[4] = {1, 1, 1, 1};
    if (MODE == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { mu[j] = p.mean[4 * chunk + j]; is[j] = p.invstd[4 * chunk + j]; }
    }
    const int t0 = split * p.tiles_per_split;
    const int t1 = min(p.ntiles, t0 + p.tiles_per_split);
    for (int t = t0 + half; t < t1; t += 2) {
        const long long row = (long long)t * 128 + r;
        if (row >= p.rows) continue;
        const float4 a = tv_ld(p.a, row, chunk);
        const float av[4] = {a.x, a.y, a.z, a.w};
        if (MODE == 1) {
            float yv[4] = {1.f, 1.f, 1.f, 1.f};
            if (p.b.base) { const float4 y = tv_ld(p.b, row, chunk); yv[0] = y.x; yv[1] = y.y; yv[2] = y.z; yv[3] = y.w; }
            const float4 z = tv_ld(p.c, row, chunk);
            const float zv[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float g = yv[j] > 0.f ? av[j] : 0.f;
                s[j] += (double)g;
                q[j] += (double)g * (double)((zv[j] - mu[j]) * is[j]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                s[j] += (double)av[j];
                if (MODE == 0) q[j] += (double)av[j] * (double)av[j];
            }
        }
    }
    __shared__ double red[256][8];
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[threadIdx.x][j] = s[j]; red[threadIdx.x][4 + j] = q[j]; }
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
#pragma unroll
            for (int j = 0; j < 8; ++j) red[threadIdx.x][j] += red[threadIdx.x + w][j];
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) {
        double *o = p.partial + ((size_t)split * p.C + 4 * chunk + threadIdx.x) * 2;
        o[0] = red[0][threadIdx.x];
        o[1] = red[0][4 + threadIdx.x];
    }
}

struct Splits { int ntiles, splits, tps; };
inline Splits plan_splits(long long rows, int chunks)
{
    Splits s;
    s.ntiles = (int)((rows + 127) / 128);
    int want = (592 + chunks - 1) / chunks;          // ~4 CTAs per SM over all chunks
    if (want < 1) want = 1;
    if (want > (s.ntiles + 1) / 2) want = (s.ntiles + 1) / 2;
    if (want < 1) want = 1;
    s.tps = (s.ntiles + want - 1) / want;
    s.splits = (s.ntiles + s.tps - 1) / s.tps;
    return s;
}
constexpr int kMaxSplits = 600;

// batch statistics -> mean / invstd (saved for the backward) + running statistics in place (nn.BatchNorm train mode:
// running = (1 - momentum) * running + momentum * batch, the variance unbiased)
__global__ void bn_finalize_kernel(const double *partial, int splits, int C, double n, float eps, float momentum,
                                   float *save_mean, float *save_invstd, float *running_mean, float *running_var)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0, q = 0;
    for (int i = 0; i < splits; ++i) { s += partial[((size_t)i * C + c) * 2]; q += partial[((size_t)i * C + c) * 2 + 1]; }
    const double mean = s / n;
    double var = q / n - mean * mean;
    if (var < 0) var = 0;
    save_mean[c] = (float)mean;
    save_invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) running_mean[c] = (float)((1.0 - momentum) * (double)running_mean[c] + momentum * mean);
    if (running_var) running_var[c] = (float)((1.0 - momentum) * (double)running_var[c] + momentum * var * (n > 1 ? n / (n - 1) : 1.0));
}

// y = relu?(z * alpha + beta') with alpha = invstd * gamma, beta' = beta - mean * alpha (torch's CPU formulation)
__global__ void bn_apply_kernel(TView z, TView y, long long rows, int chunks, const float *mean, const float *invstd,
                                const float *gamma, const float *beta, int relu)
{
    const long long total = (long long)((rows + 127) / 128) * chunks * 128;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e & 127);
        const long long pc = e >> 7;
        const int chunk = (int)(pc % chunks);
        const long long row = (pc / chunks) * 128 + r;
        float4 v = tv_ld(z, row, chunk);
        float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = 4 * chunk + j;
            const float al = invstd[c] * gamma[c];
            const float be = beta[c] - mean[c] * al;
            float t = fmaf(o[j], al, be);
            if (relu) t = t > 0.f ? t : 0.f;
            o[j] = row < rows ? t : 0.f;
        }
        tv_st(y, row, chunk, make_float4(o[0], o[1], o[2], o[3]));
    }
}

__global__ void bn_bwd_finalize_kernel(const double *partial, int splits, int C, float *dgamma, float *dbeta)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0, q = 0;
    for (int i = 0; i < splits; ++i) { s += partial[((size_t)i * C + c) * 2]; q += partial[((size_t)i * C + c) * 2 + 1]; }
    dbeta[c] = (float)s;
    dgamma[c] = (float)q;
}

// dz = (g - dbeta / n - xhat * dgamma / n) * gamma * invstd, g = dy * [y > 0]; rows past the end are zeroed so that the
// weight-gradient GEMM may run over whole tiles
__global__ void bn_bwd_apply_kernel(TView dy, TView y, TView z, TView dz, long long rows, int chunks, const float *mean,
                                    const float *invstd, const float *gamma, const float *dgamma, const float *dbeta, float inv_n)
{
    const long long total = (long long)((rows + 127) / 128) * chunks * 128;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e & 127);
        const long long pc = e >> 7;
        const int chunk = (int)(pc % chunks);
        const long long row = (pc / chunks) * 128 + r;
        float o[4] = {0.f, 0.f, 0.f, 0.f};
        if (row < rows) {
            const float4 d = tv_ld(dy, row, chunk);
            const float4 zz = tv_ld(z, row, chunk);
            float yv[4] = {1.f, 1.f, 1.f, 1.f};
            if (y.base) { const float4 yy = tv_ld(y, row, chunk); yv[0] = yy.x; yv[1] = yy.y; yv[2] = yy.z; yv[3] = yy.w; }
            const float dv[4] = {d.x, d.y, d.z, d.w}, zv[4] = {zz.x, zz.y, zz.z, zz.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = 4 * chunk + j;
                const float g = yv[j] > 0.f ? dv[j] : 0.f;
                const float xh = (zv[j] - mean[c]) * invstd[c];
                o[j] = (g - dbeta[c] * inv_n - xh * dgamma[c] * inv_n) * gamma[c] * invstd[c];
            }
        }
        tv_st(dz, row, chunk, make_float4(o[0], o[1], o[2], o[3]));
    }
}

__global__ void colsum_finalize_kernel(const double *partial, int splits, int C, int cout, float *out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cout) return;
    double s = 0;
    for (int i = 0; i < splits; ++i) s += partial[((size_t)i * C + c) * 2];
    out[c] = (float)s;
}

// ------------------------------------------------------------------------------------------------
// weight gradient: dW[n][k] = sum_r dZ[r][n] * X[r][k], X = [A1 | A2] (feature-propagation concat).  Split-K over row
// ranges: grid (n tiles, k tiles, splits), 64 x 64 outputs per CTA, 32 rows per smem stage, 4 x 4 outputs per thread;
// the partial tiles are summed in split order by wgrad_reduce_kernel (deterministic).
// ------------------------------------------------------------------------------------------------
struct WgradArgs {
    TView dz, a1, a2;
    int k1chunks, k2chunks;
    long long rows;
    int ntiles, tiles_per_split;
    float *partial;             // [splits][npad][kpad]
    int npad, kpad;
    int dz_chunks;              // padded width of dz / 4 (tile columns beyond it read as zero)
};

__global__ void __launch_bounds__(256) wgrad_kernel(WgradArgs p)
{
    __shared__ __align__(16) float dzs[32][68];
    __shared__ __align__(16) float xs[32][68];
    const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64, split = blockIdx.z;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int t0 = split * p.tiles_per_split, t1 = min(p.ntiles, t0 + p.tiles_per_split);
    const int kchunks = p.k1chunks + p.k2chunks;
    for (int t = t0; t < t1; ++t) {
        for (int sub = 0; sub < 4; ++sub) {
            const long long rbase = (long long)t * 128 + sub * 32;
            __syncthreads();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int e = threadIdx.x + h * 256;          // 0..511 = 16 chunks x 32 rows
                const int cc = e >> 5, rr = e & 31;
                const long long row = rbase + rr;
                float4 d = make_float4(0.f, 0.f, 0.f, 0.f), x = d;
                if (row < p.rows) {
                    const int nc = (n0 >> 2) + cc;
                    if (nc < p.dz_chunks) d = tv_ld(p.dz, row, nc);
                    const int kc = (k0 >> 2) + cc;
                    if (kc < kchunks) x = kc < p.k1chunks ? tv_ld(p.a1, row, kc) : tv_ld(p.a2, row, kc - p.k1chunks);
                }
                *reinterpret_cast<float4 *>(&dzs[rr][cc * 4]) = d;
                *reinterpret_cast<float4 *>(&xs[rr][cc * 4]) = x;
            }
            __syncthreads();
#pragma unroll 8
            for (int rr = 0; rr < 32; ++rr) {
                const float4 d = *reinterpret_cast<const float4 *>(&dzs[rr][ty * 4]);
                const float4 x = *reinterpret_cast<const float4 *>(&xs[rr][tx * 4]);
                const float dv[4] = {d.x, d.y, d.z, d.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], xv[j], acc[i][j]);
            }
        }
    }
    float *o = p.partial + (size_t)split * p.npad * p.kpad;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= p.npad) continue;
        const int k = k0 + tx * 4;
        if (k < p.kpad) *reinterpret_cast<float4 *>(o + (size_t)n * p.kpad + k) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
}

__global__ void wgrad_reduce_kernel(const float *partial, int splits, int npad, int kpad, int cout, int cin, float *dW,
                                    int accumulate)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= cout * cin) return;
    const int n = idx / cin, k = idx - n * cin;
    float s = 0.f;
    for (int i = 0; i < splits; ++i) s += partial[((size_t)i * npad + n) * kpad + k];
    dW[idx] = accumulate ? dW[idx] + s : s;
}

// ------------------------------------------------------------------------------------------------
// weighted NLL (pointnet2_sem_seg.py:47): loss = - sum_i w[y_i] logp[i][y_i] / sum_i w[y_i]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nll_partial_kernel(const float *logp, const long long *labels, const float *weight,
                                                          long long rows, int ncls, double *partial)
{
    double num = 0, den = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (long long)gridDim.x * blockDim.x) {
        const long long y = labels[i];
        if (y < 0 || y >= ncls) continue;                 // (ignore_index semantics for out-of-range labels)
        const float w = weight ? weight[y] : 1.f;
        num -= (double)w * (double)logp[i * ncls + y];
        den += (double)w;
    }
    __shared__ double red[256][2];
    red[threadIdx.x][0] = num; red[threadIdx.x][1] = den;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) { red[threadIdx.x][0] += red[threadIdx.x + w][0]; red[threadIdx.x][1] += red[threadIdx.x + w][1]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { partial[2 * blockIdx.x] = red[0][0]; partial[2 * blockIdx.x + 1] = red[0][1]; }
}
__global__ void nll_finalize_kernel(const double *partial, int nblocks, float *loss, float *wsum)
{
    double num = 0, den = 0;
    for (int i = 0; i < nblocks; ++i) { num += partial[2 * i]; den += partial[2 * i + 1]; }
    *loss = (float)(num / den);
    *wsum = (float)den;
}
__global__ void nll_backward_kernel(const long long *labels, const float *weight, long long rows, int ncls, const float *gout,
                                    const float *wsum, float *dlogp)
{
    const long long total = rows * ncls;
    const float g = gout ? *gout : 1.f;
    const float inv = 1.f / *wsum;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / ncls;
        const int c = (int)(e - i * ncls);
        const long long y = labels[i];
        float v = 0.f;
        if (y == c) v = -(weight ? weight[y] : 1.f) * inv * g;
        dlogp[e] = v;
    }
}

// x *= m * scale on T-layout tensors of the same shape (dropout forward and backward)
__global__ void tl_mul_kernel(TView x, TView m, long long rows, int chunks, float scale)
{
    const long long total = (long long)((rows + 127) / 128) * chunks * 128;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e & 127);
        const long long pc = e >> 7;
        const int chunk = (int)(pc % chunks);
        const long long row = (pc / chunks) * 128 + r;
        float4 a = tv_ld(x, row, chunk);
        const float4 b = tv_ld(m, row, chunk);
        a.x *= b.x * scale; a.y *= b.y * scale; a.z *= b.z * scale; a.w *= b.w * scale;
        tv_st(x, row, chunk, a);
    }
}

// torch.optim.Adam (single-tensor formulation of torch/optim/adam.py, amsgrad off, maximize off):
//   g += wd * p;  m = m + (g - m) * (1 - b1)  [lerp];  v = v * b2 + g * g * (1 - b2);
//   p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
__global__ void adam_kernel(float *p, const float *g, float *m, float *v, long long n, float lr, float b1, float b2, float eps,
                            float wd, float bc1, float bc2_sqrt)
{
    const float step_size = lr / bc1;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float gi = g[i];
        const float pi = p[i];
        if (wd != 0.f) gi = fmaf(wd, pi, gi);
        float mi = m[i];
        mi = fmaf(gi - mi, 1.f - b1, mi);
        float vi = v[i] * b2;
        vi = fmaf(gi * (1.f - b2), gi, vi);
        m[i] = mi; v[i] = vi;
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        p[i] = pi - step_size * (mi / denom);
    }
}

// W [cout][cin] row-major (device) -> the two packed operand layouts of a psg_mlp (exact + TF32-compensated copies)
__global__ void repack_kernel(const float *w, const float *b, int cout, int cin, int kpad, int npad, int nwf, int nwb,
                              float *wf, float *wb, float *wf_c, float *wb_c, float *bias, float comp)
{
    const long long nf = (long long)kpad * nwf, nb = (long long)npad * nwb;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nf + nb + nwf; e += (long long)gridDim.x * blockDim.x) {
        if (e < nf) {
            const int q = (int)(e & 3);
            const long long t = e >> 2;
            const int n = (int)(t % nwf), kc = (int)(t / nwf);
            const int k = 4 * kc + q;
            const float v = (n < cout && k < cin) ? w[(size_t)n * cin + k] : 0.f;
            wf[e] = v;
            unsigned u = __float_as_uint(v * (1.f + comp));
            u = (u + 0x1000u) & 0xffffe000u;
            wf_c[e] = __uint_as_float(u);
        } else if (e < nf + nb) {
            const long long f = e - nf;
            const int q = (int)(f & 3);
            const long long t = f >> 2;
            const int k = (int)(t % nwb), nc = (int)(t / nwb);
            const int n = 4 * nc + q;
            const float v = (n < cout && k < cin) ? w[(size_t)n * cin + k] : 0.f;
            wb[f] = v;
            unsigned u = __float_as_uint(v * (1.f + comp));
            u = (u + 0x1000u) & 0xffffe000u;
            wb_c[f] = __uint_as_float(u);
        } else {
            const int n = (int)(e - nf - nb);
            bias[n] = (b && n < cout) ? b[n] : 0.f;
        }
    }
}

inline int ew_grid(long long total) { long long g = (total + 255) / 256; return (int)(g > 148 * 16 ? 148 * 16 : (g < 1 ? 1 : g)); }

}  // namespace

int psg_repack_weights(const float *w, const float *b, int cout, int cin, int kpad, int npad, int nwf, int nwb, float *wf,
                       float *wb, float *wf_c, float *wb_c, float *bias, float comp, cudaStream_t st)
{
    const long long total = (long long)kpad * nwf + (long long)npad * nwb + nwf;
    repack_kernel<<<ew_grid(total), 256, 0, st>>>(w, b, cout, cin, kpad, npad, nwf, nwb, wf, wb, wf_c, wb_c, bias, comp);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" size_t psg_bn_workspace(int C)
{
    return C > 0 ? (size_t)kMaxSplits * ((C + 3) / 4 * 4) * 2 * sizeof(double) : 0;
}

extern "C" int psg_bn_train_forward(const float *z_base, int z_wchunks, int64_t rows, int C, const float *gamma,
                                    const float *beta, float *running_mean, float *running_var, float momentum, float eps,
                                    float *y_base, int y_wchunks, int relu, float *save_mean, float *save_invstd,
                                    void *workspace, size_t workspace_bytes, psg_stream_t stream)
{
    if (!z_base || !y_base || !gamma || !beta || !save_mean || !save_invstd || !workspace || rows <= 0 || C <= 0 || C % 4) return PSG_EINVAL;
    if (4 * z_wchunks < C || 4 * y_wchunks < C) return PSG_EINVAL;
    if (workspace_bytes < psg_bn_workspace(C)) return PSG_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int chunks = C / 4;
    Splits sp = plan_splits(rows, chunks);
    if (sp.splits > kMaxSplits) return PSG_EUNSUPPORTED;
    ColRedArgs a;
    a.a = mkv(z_base, z_wchunks, 0); a.b = a.c = TView{nullptr, 0, 0}; a.mean = a.invstd = nullptr;
    a.rows = rows; a.ntiles = sp.ntiles; a.tiles_per_split = sp.tps; a.partial = (double *)workspace; a.C = C;
    colred_kernel<0><<<dim3(chunks, sp.splits), 256, 0, st>>>(a);
    PSG_LAUNCH_CHECK();
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>((const double *)workspace, sp.splits, C, (double)rows, eps, momentum,
                                                        save_mean, save_invstd, running_mean, running_var);
    PSG_LAUNCH_CHECK();
    const long long total = (long long)sp.ntiles * chunks * 128;
    bn_apply_kernel<<<ew_grid(total), 256, 0, st>>>(mkv(z_base, z_wchunks, 0), mkv(y_base, y_wchunks, 0), rows, chunks, save_mean,
                                                    save_invstd, gamma, beta, relu);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" int psg_bn_train_backward(const float *dy_base, int dy_wchunks, const float *y_base, int y_wchunks,
                                     const float *z_base, int z_wchunks, int64_t rows, int C, const float *gamma,
                                     const float *save_mean, const float *save_invstd, float *dgamma, float *dbeta,
                                     float *dz_base, int dz_wchunks, void *workspace, size_t workspace_bytes,
                                     psg_stream_t stream)
{
    if (!dy_base || !z_base || !gamma || !save_mean || !save_invstd || !dgamma || !dbeta || !dz_base || !workspace || rows <= 0 ||
        C <= 0 || C % 4)
        return PSG_EINVAL;
    if (4 * dy_wchunks < C || 4 * z_wchunks < C || 4 * dz_wchunks < C || (y_base && 4 * y_wchunks < C)) return PSG_EINVAL;
    if (workspace_bytes < psg_bn_workspace(C)) return PSG_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int chunks = C / 4;
    Splits sp = plan_splits(rows, chunks);
    if (sp.splits > kMaxSplits) return PSG_EUNSUPPORTED;
    ColRedArgs a;
    a.a = mkv(dy_base, dy_wchunks, 0); a.b = mkv(y_base, y_wchunks, 0); a.c = mkv(z_base, z_wchunks, 0);
    a.mean = save_mean; a.invstd = save_invstd;
    a.rows = rows; a.ntiles = sp.ntiles; a.tiles_per_split = sp.tps; a.partial = (double *)workspace; a.C = C;
    colred_kernel<1><<<dim3(chunks, sp.splits), 256, 0, st>>>(a);
    PSG_LAUNCH_CHECK();
    bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>((const double *)workspace, sp.splits, C, dgamma, dbeta);
    PSG_LAUNCH_CHECK();
    const long long total = (long long)sp.ntiles * chunks * 128;
    bn_bwd_apply_kernel<<<ew_grid(total), 256, 0, st>>>(mkv(dy_base, dy_wchunks, 0), mkv(y_base, y_wchunks, 0), mkv(z_base, z_wchunks, 0),
                                                        mkv(dz_base, dz_wchunks, 0), rows, chunks, save_mean, save_invstd, gamma,
                                                        dgamma, dbeta, (float)(1.0 / (double)rows));
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" size_t psg_wgrad_workspace(int cout, int cin, int64_t rows)
{
    if (cout <= 0 || cin <= 0 || rows <= 0) return 0;
    const int npad = round_up(cout, 64), kpad = round_up(cin, 64);
    const size_t wg = (size_t)kMaxSplits * npad * kpad * sizeof(float);
    const size_t cs = psg_bn_workspace(round_up(cout, 16));
    // the split count is bounded by the tile count, so small problems need far less than the cap
    const long long ntiles = (rows + 127) / 128;
    const size_t wg2 = (size_t)(ntiles < kMaxSplits ? ntiles : kMaxSplits) * npad * kpad * sizeof(float);
    return (wg2 < wg ? wg2 : wg) + cs + 1024;
}

extern "C" int psg_conv_wgrad(const float *dz_base, int dz_wchunks, int cout, const float *a1_base, int a1_wchunks, int a1_c0,
                              int k1, const float *a2_base, int a2_wchunks, int a2_c0, int k2, int64_t rows, float *dW,
                              float *db, int accumulate, void *workspace, size_t workspace_bytes, psg_stream_t stream)
{
    if (!dz_base || !a1_base || !dW || !workspace || cout <= 0 || k1 <= 0 || k2 < 0 || rows <= 0) return PSG_EINVAL;
    if (k2 > 0 && (!a2_base || k1 % 4)) return PSG_EINVAL;
    // every view must hold the columns it is read for: dz the cout columns of dW / db, A1 (A2) k1 (k2) columns from a1_c0
    // (a2_c0) on -- a narrower view would read into the next row tile
    if (4 * dz_wchunks < cout || a1_c0 < 0 || a1_c0 + (k1 + 3) / 4 > a1_wchunks) return PSG_EINVAL;
    if (k2 > 0 && (a2_c0 < 0 || a2_c0 + (k2 + 3) / 4 > a2_wchunks)) return PSG_EINVAL;
    if (workspace_bytes < psg_wgrad_workspace(cout, k1 + k2, rows)) return PSG_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int cin = k1 + k2;
    WgradArgs p;
    p.dz = mkv(dz_base, dz_wchunks, 0); p.a1 = mkv(a1_base, a1_wchunks, a1_c0); p.a2 = mkv(a2_base, a2_wchunks, a2_c0);
    p.k1chunks = (k1 + 3) / 4; p.k2chunks = (k2 + 3) / 4;
    p.rows = rows; p.ntiles = (int)((rows + 127) / 128);
    p.npad = round_up(cout, 64); p.kpad = round_up(cin, 64);
    p.dz_chunks = dz_wchunks;
    const int nt = p.npad / 64, kt = p.kpad / 64;
    int splits = (592 + nt * kt - 1) / (nt * kt);
    if (splits > p.ntiles) splits = p.ntiles;
    if (splits > kMaxSplits) splits = kMaxSplits;
    if (splits < 1) splits = 1;
    p.tiles_per_split = (p.ntiles + splits - 1) / splits;
    splits = (p.ntiles + p.tiles_per_split - 1) / p.tiles_per_split;
    p.partial = (float *)workspace;
    wgrad_kernel<<<dim3(nt, kt, splits), 256, 0, st>>>(p);
    PSG_LAUNCH_CHECK();
    const int total = cout * cin;
    wgrad_reduce_kernel<<<(total + 255) / 256, 256, 0, st>>>((const float *)workspace, splits, p.npad, p.kpad, cout, cin, dW, accumulate);
    PSG_LAUNCH_CHECK();
    if (db) {
        const int C = round_up(cout, 4);
        const int chunks = C / 4;
        Splits sp = plan_splits(rows, chunks);
        double *part = (double *)((char *)workspace + (((size_t)splits * p.npad * p.kpad * sizeof(float) + 1023) & ~(size_t)1023));
        ColRedArgs a;
        a.a = mkv(dz_base, dz_wchunks, 0); a.b = a.c = TView{nullptr, 0, 0}; a.mean = a.invstd = nullptr;
        a.rows = rows; a.ntiles = sp.ntiles; a.tiles_per_split = sp.tps; a.partial = part; a.C = C;
        colred_kernel<2><<<dim3(chunks, sp.splits), 256, 0, st>>>(a);
        PSG_LAUNCH_CHECK();
        colsum_finalize_kernel<<<(cout + 127) / 128, 128, 0, st>>>(part, sp.splits, C, cout, db);
        PSG_LAUNCH_CHECK();
    }
    return PSG_OK;
}

extern "C" int psg_log_softmax_rows(const float *z_base, int z_wchunks, int64_t rows, int ncls, float *logp, psg_stream_t stream)
{
    if (!z_base || !logp || rows <= 0 || ncls < 2 || ncls > 16 || 4 * z_wchunks < ncls) return PSG_EINVAL;
    return psg_head_logsoftmax(mkv(z_base, z_wchunks, 0), rows, ncls, logp, (cudaStream_t)stream);
}

extern "C" int psg_dlogits_from_dlogp(const float *z_base, int z_wchunks, const float *dlogp, int64_t rows, int ncls,
                                      float *dz_base, int dz_wchunks, psg_stream_t stream)
{
    // dz: all 16 columns of the row are written (zeros past ncls)
    if (!z_base || !dlogp || !dz_base || rows <= 0 || ncls < 2 || ncls > 16 || 4 * z_wchunks < ncls || dz_wchunks < 4)
        return PSG_EINVAL;
    return psg_dz_from_dlogp(mkv(z_base, z_wchunks, 0), dlogp, rows, ncls, mkv(dz_base, dz_wchunks, 0), (cudaStream_t)stream);
}

extern "C" size_t psg_nll_workspace(void) { return (size_t)2 * 1024 * sizeof(double); }

extern "C" int psg_nll_loss(const float *logp, const int64_t *labels, const float *weight, int64_t rows, int ncls, float *loss,
                            float *wsum, void *workspace, size_t workspace_bytes, psg_stream_t stream)
{
    if (!logp || !labels || !loss || !wsum || !workspace || rows <= 0 || ncls < 2) return PSG_EINVAL;
    if (workspace_bytes < psg_nll_workspace()) return PSG_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    int nb = (int)((rows + 255) / 256);
    if (nb > 1024) nb = 1024;
    nll_partial_kernel<<<nb, 256, 0, st>>>(logp, (const long long *)labels, weight, rows, ncls, (double *)workspace);
    PSG_LAUNCH_CHECK();
    nll_finalize_kernel<<<1, 1, 0, st>>>((const double *)workspace, nb, loss, wsum);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" int psg_nll_loss_backward(const int64_t *labels, const float *weight, int64_t rows, int ncls, const float *grad_out,
                                     const float *wsum, float *dlogp, psg_stream_t stream)
{
    if (!labels || !wsum || !dlogp || rows <= 0 || ncls < 2) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    nll_backward_kernel<<<ew_grid(rows * ncls), 256, 0, st>>>((const long long *)labels, weight, rows, ncls, grad_out, wsum, dlogp);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" int psg_tl_mul(float *x_base, int x_wchunks, const float *m_base, int m_wchunks, int64_t rows, int C, float scale,
                          psg_stream_t stream)
{
    if (!x_base || !m_base || rows <= 0 || C <= 0 || C % 4 || 4 * x_wchunks < C || 4 * m_wchunks < C) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)((rows + 127) / 128) * (C / 4) * 128;
    tl_mul_kernel<<<ew_grid(total), 256, 0, st>>>(mkv(x_base, x_wchunks, 0), mkv(m_base, m_wchunks, 0), rows, C / 4, scale);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

extern "C" int psg_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int step, psg_stream_t stream)
{
    if (!param || !grad || !exp_avg || !exp_avg_sq || n <= 0 || step < 1) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    adam_kernel<<<ew_grid(n), 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, (float)bc1,
                                            (float)sqrt(bc2));
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
