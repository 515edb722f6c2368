// neighbors.cu -- ball query, 3-NN (+ inverse-distance weights) and the dense square_distance op.
// Reference: PointNet/models/pointnet_util.py:19-40 (square_distance), :87-107 (query_ball_point),
// :301-307 (3-NN + weights inside PointNetFeaturePropagation.forward).
//
// The reference materialises [B,S,N] distance and index tensors and fully sorts them.  Here the
// cloud is staged once per CTA in shared memory (SoA + |p|^2) and
//   * ball query: one warp per centroid scans the cloud 32 points at a time, compacts the in-radius
//     lanes with a ballot/popc prefix, stops as soon as every radius has nsample hits, and pads with
//     the first hit.  Up to two radii (the MSG pair) share one scan.
//   * 3-NN: one thread per fine point keeps a register top-3 over the (broadcast) coarse points;
//     strict '<' keeps the lowest index among equal distances.
// Distances are computed in the oracle's exact op order so the indices are bit-identical.
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

constexpr int kBallChunk = 4096;   // points staged per pass: 4 arrays * 16 KB = 64 KB

template <int NR>
__global__ void __launch_bounds__(1024)
ball_query_kernel(const float *__restrict__ xyz, long long cloud_stride, int nclouds, int N,
                  const float *__restrict__ new_xyz, int S, float r2a, float r2b, int Ka, int Kb,
                  int *__restrict__ outa, int *__restrict__ outb)
{
    extern __shared__ float smem[];
    float *sx = smem, *sy = sx + kBallChunk, *sz = sy + kBallChunk, *sn = sz + kBallChunk;
    const int p = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    const int s = blockIdx.x * nwarps + warp;
    const float *cloud = xyz + (long long)(p % nclouds) * cloud_stride;
    const bool active = s < S;

    float qx = 0.f, qy = 0.f, qz = 0.f, qn = 0.f;
    if (active) {
        const float *q = new_xyz + ((long long)p * S + s) * 3;
        qx = q[0]; qy = q[1]; qz = q[2];
        qn = psg_sqnorm(qx, qy, qz);
    }
    int *oa = outa + ((long long)p * S + (active ? s : 0)) * Ka;
    int *ob = (NR == 2) ? outb + ((long long)p * S + (active ? s : 0)) * Kb : nullptr;
    int cnta = 0, cntb = 0, firsta = -1, firstb = -1;
    bool done = !active;

    for (int base0 = 0; base0 < N; base0 += kBallChunk) {
        const int n = min(kBallChunk, N - base0);
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const float *c = cloud + (long long)(base0 + i) * 3;
            float x = c[0], y = c[1], z = c[2];
            sx[i] = x; sy[i] = y; sz[i] = z; sn[i] = psg_sqnorm(x, y, z);
        }
        __syncthreads();
        if (done) continue;
        for (int b = 0; b < n; b += 32) {
            const int i = b + lane;
            bool ha = false, hb = false;
            if (i < n) {
                float d = psg_sqdist(qx, qy, qz, qn, sx[i], sy[i], sz[i], sn[i]);
                ha = !(d > r2a);
                if (NR == 2) hb = !(d > r2b);
            }
            unsigned ma = __ballot_sync(0xffffffffu, ha && cnta < Ka);
            if (ma) {
                if (firsta < 0) firsta = base0 + b + __ffs(ma) - 1;
                int pos = cnta + __popc(ma & ((1u << lane) - 1u));
                if (ha && pos < Ka) oa[pos] = base0 + i;
                cnta = min(Ka, cnta + __popc(ma));
            }
            if (NR == 2) {
                unsigned mb = __ballot_sync(0xffffffffu, hb && cntb < Kb);
                if (mb) {
                    if (firstb < 0) firstb = base0 + b + __ffs(mb) - 1;
                    int pos = cntb + __popc(mb & ((1u << lane) - 1u));
                    if (hb && pos < Kb) ob[pos] = base0 + i;
                    cntb = min(Kb, cntb + __popc(mb));
                }
            }
            if (cnta >= Ka && (NR == 1 || cntb >= Kb)) { done = true; break; }
        }
    }
    if (active) {
        // pointnet_util.py:104-106: unfilled slots take the first hit (N if there was none)
        const int fa = firsta < 0 ? N : firsta;
        for (int k = cnta + lane; k < Ka; k += 32) oa[k] = fa;
        if (NR == 2) {
            const int fb = firstb < 0 ? N : firstb;
            for (int k = cntb + lane; k < Kb; k += 32) ob[k] = fb;
        }
    }
}

constexpr int kNnChunk = 2048;
constexpr int kNnQ = 2;             // fine points per thread: one LDS.128 of a coarse point serves both

// running top-3 of (d, j): strict '<' keeps the lowest index among equal distances (candidates arrive in
// ascending index order), which is what the oracle pins for the reference's sort (SURVEY.md App. B)
__device__ __forceinline__ void top3_push(float d, int jj, float &d0, float &d1, float &d2, int &i0, int &i1, int &i2)
{
    if (d < d2 || i2 < 0) {
        if (d < d1 || i1 < 0) {
            d2 = d1; i2 = i1;
            if (d < d0 || i0 < 0) { d1 = d0; i1 = i0; d0 = d; i0 = jj; }
            else { d1 = d; i1 = jj; }
        } else { d2 = d; i2 = jj; }
    }
}

__global__ void __launch_bounds__(256)
three_nn_kernel(const float *__restrict__ xyz1, long long stride1, int nclouds1, int N,
                const float *__restrict__ xyz2, int S,
                int *__restrict__ idx, float *__restrict__ wout, float *__restrict__ d2out)
{
    __shared__ float4 sp[kNnChunk];             // coarse points (x, y, z, |p|^2)
    const int p = blockIdx.y;
    const float *fine = xyz1 + (long long)(p % nclouds1) * stride1;
    const float *coarse = xyz2 + (long long)p * S * 3;
    int qi[kNnQ];
    float qx[kNnQ], qy[kNnQ], qz[kNnQ], qn[kNnQ];
    float d0[kNnQ], d1[kNnQ], d2[kNnQ];
    int i0[kNnQ], i1[kNnQ], i2[kNnQ];
#pragma unroll
    for (int u = 0; u < kNnQ; ++u) {
        qi[u] = (blockIdx.x * kNnQ + u) * blockDim.x + threadIdx.x;
        qx[u] = qy[u] = qz[u] = qn[u] = 0.f;
        if (qi[u] < N) {
            qx[u] = fine[3 * qi[u]]; qy[u] = fine[3 * qi[u] + 1]; qz[u] = fine[3 * qi[u] + 2];
            qn[u] = psg_sqnorm(qx[u], qy[u], qz[u]);
        }
        d0[u] = d1[u] = d2[u] = INFINITY;
        i0[u] = i1[u] = i2[u] = -1;
    }
    for (int base = 0; base < S; base += kNnChunk) {
        const int n = min(kNnChunk, S - base);
        __syncthreads();
        for (int j = threadIdx.x; j < n; j += blockDim.x) {
            const float *c = coarse + (long long)(base + j) * 3;
            const float x = c[0], y = c[1], z = c[2];
            sp[j] = make_float4(x, y, z, psg_sqnorm(x, y, z));
        }
        __syncthreads();
        for (int j = 0; j < n; ++j) {
            const float4 c = sp[j];
#pragma unroll
            for (int u = 0; u < kNnQ; ++u) {
                const float d = psg_sqdist(qx[u], qy[u], qz[u], qn[u], c.x, c.y, c.z, c.w);
                top3_push(d, base + j, d0[u], d1[u], d2[u], i0[u], i1[u], i2[u]);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < kNnQ; ++u) {
        if (qi[u] >= N) continue;
        const long long o = ((long long)p * N + qi[u]) * 3;
        idx[o] = i0[u]; idx[o + 1] = i1[u]; idx[o + 2] = i2[u];
        // pointnet_util.py:305-307: recip = 1/(d+1e-8); w = recip / (r0 + r1 + r2)
        const float r0 = __fdiv_rn(1.0f, __fadd_rn(d0[u], 1e-8f));
        const float r1 = __fdiv_rn(1.0f, __fadd_rn(d1[u], 1e-8f));
        const float r2 = __fdiv_rn(1.0f, __fadd_rn(d2[u], 1e-8f));
        const float nrm = __fadd_rn(__fadd_rn(r0, r1), r2);
        if (wout) { wout[o] = __fdiv_rn(r0, nrm); wout[o + 1] = __fdiv_rn(r1, nrm); wout[o + 2] = __fdiv_rn(r2, nrm); }
        if (d2out) { d2out[o] = d0[u]; d2out[o + 1] = d1[u]; d2out[o + 2] = d2[u]; }
    }
}


// ---- 3-NN through a uniform grid over the coarse cloud ---------------------------------------------------
// Same results as three_nn_kernel, bit for bit: every candidate's distance is computed with the same
// expansion-form arithmetic and the top-3 is kept under the total order (distance, index), so the order in
// which candidates are visited does not matter.  The grid only decides WHICH candidates are visited: rings of
// cells around the query's cell, until the third-best distance found so far is below the squared distance to
// everything not visited yet -- minus a margin that covers the rounding error of the expansion formula
// (|computed - true| <= ~1e-6 * max|p|^2; a query that cannot prove the bound simply visits more rings, up to
// the whole grid).  ~70 candidates per query instead of 1024 at fp1.
constexpr int kNgMaxS = 2048, kNgMaxCells = 2048, kNgQ = 1024;     // coarse points, cells, queries per CTA

__device__ __forceinline__ bool nn_less(float d, int j, float D, int I) { return I < 0 || d < D || (d == D && j < I); }
__device__ __forceinline__ void top3_push_lex(float d, int jj, float &d0, float &d1, float &d2, int &i0, int &i1, int &i2)
{
    if (nn_less(d, jj, d2, i2)) {
        if (nn_less(d, jj, d1, i1)) {
            d2 = d1; i2 = i1;
            if (nn_less(d, jj, d0, i0)) { d1 = d0; i1 = i0; d0 = d; i0 = jj; }
            else { d1 = d; i1 = jj; }
        } else { d2 = d; i2 = jj; }
    }
}

__global__ void __launch_bounds__(256)
three_nn_grid_kernel(const float *__restrict__ xyz1, long long stride1, int nclouds1, int N,
                     const float *__restrict__ xyz2, int S,
                     int *__restrict__ idx, float *__restrict__ wout, float *__restrict__ d2out)
{
    extern __shared__ __align__(16) unsigned char nn_sm[];
    float4 *sp = reinterpret_cast<float4 *>(nn_sm);                  // [S] points sorted by cell (x, y, z, |p|^2)
    int *sid = reinterpret_cast<int *>(sp + S);                      // [S] their original indices
    int *cstart = sid + S;                                           // [cells + 1]
    int *ccnt = cstart + kNgMaxCells + 1;                            // [cells] fill cursors
    __shared__ float red[6][8];
    __shared__ float sb[8];                                          // bbox min (3), cell size, margin
    __shared__ int sdim[4];

    const int p = blockIdx.y, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float *fine = xyz1 + (long long)(p % nclouds1) * stride1;
    const float *coarse = xyz2 + (long long)p * S * 3;

    // ---- bounding box of the coarse cloud ----
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    bool fin = true;
    for (int j = t; j < S; j += 256) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = coarse[3 * j + a];
            mn[a] = fminf(mn[a], v); mx[a] = fmaxf(mx[a], v);
            fin = fin && isfinite(v);                                // fminf / fmaxf skip a NaN: count it here
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
        if (lane == 0) { red[a][warp] = mn[a]; red[3 + a][warp] = mx[a]; }
    }
    const bool all_finite = __syncthreads_and(fin);
    if (t == 0) {
        float lo[3], hi[3], ext[3];
        for (int a = 0; a < 3; ++a) {
            lo[a] = red[a][0]; hi[a] = red[3 + a][0];
            for (int w = 1; w < 8; ++w) { lo[a] = fminf(lo[a], red[a][w]); hi[a] = fmaxf(hi[a], red[3 + a][w]); }
            ext[a] = fmaxf(hi[a] - lo[a], 1e-6f);
        }
        // about two points per cell; at most 16 cells per axis and kNgMaxCells in total
        float h = cbrtf(ext[0] * ext[1] * ext[2] * 2.0f / (float)S);
        h = fmaxf(h, fmaxf(ext[0], fmaxf(ext[1], ext[2])) / 16.0f);
        int d[3];
        for (int a = 0; a < 3; ++a) { d[a] = (int)(ext[a] / h) + 1; d[a] = d[a] > 16 ? 16 : d[a]; }
        while (d[0] * d[1] * d[2] > kNgMaxCells) { h *= 1.26f; for (int a = 0; a < 3; ++a) { d[a] = (int)(ext[a] / h) + 1; d[a] = d[a] > 16 ? 16 : d[a]; } }
        float m2 = 0.f;
        for (int a = 0; a < 3; ++a) { const float v = fmaxf(fabsf(lo[a]), fabsf(hi[a])); m2 += v * v; }
        if (!all_finite) m2 = INFINITY;                                  // every query scans (below)
        sb[0] = lo[0]; sb[1] = lo[1]; sb[2] = lo[2]; sb[3] = h; sb[4] = m2;            // m2 >= |p|^2 of every coarse point
        sdim[0] = d[0]; sdim[1] = d[1]; sdim[2] = d[2]; sdim[3] = d[0] * d[1] * d[2];
    }
    __syncthreads();
    const float lox = sb[0], loy = sb[1], loz = sb[2], h = sb[3], m2c = sb[4], inv_h = 1.0f / h;
    const int nx = sdim[0], ny = sdim[1], nz = sdim[2], ncell = sdim[3];
    auto cell_of = [&](float x, float y, float z, int &cx, int &cy, int &cz) {
        cx = min(max((int)floorf((x - lox) * inv_h), 0), nx - 1);
        cy = min(max((int)floorf((y - loy) * inv_h), 0), ny - 1);
        cz = min(max((int)floorf((z - loz) * inv_h), 0), nz - 1);
    };
    // ---- counting sort of the coarse points by cell ----
    for (int c = t; c <= ncell; c += 256) { cstart[c] = 0; if (c < ncell) ccnt[c] = 0; }
    __syncthreads();
    for (int j = t; j < S; j += 256) {
        int cx, cy, cz;
        cell_of(coarse[3 * j], coarse[3 * j + 1], coarse[3 * j + 2], cx, cy, cz);
        atomicAdd(&cstart[(cz * ny + cy) * nx + cx + 1], 1);
    }
    __syncthreads();
    if (warp == 0) {                                     // inclusive scan of cstart[1..ncell] by one warp
        int carry = 0;
        for (int base = 1; base <= ncell; base += 32) {
            const int c = base + lane;
            int v = c <= ncell ? cstart[c] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += y; }
            if (c <= ncell) cstart[c] = v + carry;
            carry += __shfl_sync(0xffffffffu, v, 31);
        }
    }
    __syncthreads();
    for (int j = t; j < S; j += 256) {
        const float x = coarse[3 * j], y = coarse[3 * j + 1], z = coarse[3 * j + 2];
        int cx, cy, cz;
        cell_of(x, y, z, cx, cy, cz);
        const int c = (cz * ny + cy) * nx + cx;
        const int pos = cstart[c] + atomicAdd(&ccnt[c], 1);
        sp[pos] = make_float4(x, y, z, psg_sqnorm(x, y, z));
        sid[pos] = j;
    }
    __syncthreads();
    // ---- queries ----
    const int q0 = blockIdx.x * kNgQ;
    for (int qi = q0 + t; qi < min(q0 + kNgQ, N); qi += 256) {
        const float qx = fine[3 * qi], qy = fine[3 * qi + 1], qz = fine[3 * qi + 2];
        const float qn = psg_sqnorm(qx, qy, qz);
        float d0 = INFINITY, d1 = INFINITY, d2 = INFINITY;
        int i0 = -1, i1 = -1, i2 = -1;
        // A non-finite query or coarse cloud, or an |p|^2 that overflows, can make distances NaN, which the (distance,
        // index) order cannot rank: such a query scans every coarse point in index order with three_nn_kernel's
        // insertion, so it returns what the exhaustive kernel returns for any input.
        const bool scan = !(qn < INFINITY && m2c < INFINITY);
        for (int j = 0; scan && j < S; ++j) {
            const float x = coarse[3 * j], y = coarse[3 * j + 1], z = coarse[3 * j + 2];
            top3_push(psg_sqdist(qx, qy, qz, qn, x, y, z, psg_sqnorm(x, y, z)), j, d0, d1, d2, i0, i1, i2);
        }
        // rounding error of the expansion formula <= ~2.4e-6 * max(|q|^2, |p|^2): a 16x safety factor
        const float margin = 4e-5f * (1.0f + fmaxf(qn, m2c));
        int cx, cy, cz;
        cell_of(qx, qy, qz, cx, cy, cz);
        const int rmax = scan ? -1 : max(max(max(cx, nx - 1 - cx), max(cy, ny - 1 - cy)), max(cz, nz - 1 - cz));
        for (int r = 0; r <= rmax; ++r) {
            for (int dz = -r; dz <= r; ++dz) {
                const int z = cz + dz;
                if (z < 0 || z >= nz) continue;
                for (int dy = -r; dy <= r; ++dy) {
                    const int y = cy + dy;
                    if (y < 0 || y >= ny) continue;
                    const bool shell = (dz == -r || dz == r || dy == -r || dy == r);
                    const int step = shell ? 1 : 2 * r;             // interior rows of the cube: only the two end cells
                    for (int dx = -r; dx <= r; dx += (step > 0 ? step : 1)) {
                        const int x = cx + dx;
                        if (x < 0 || x >= nx) continue;
                        const int c = (z * ny + y) * nx + x;
                        for (int e = cstart[c]; e < cstart[c + 1]; ++e) {
                            const float4 cp = sp[e];
                            const float d = psg_sqdist(qx, qy, qz, qn, cp.x, cp.y, cp.z, cp.w);
                            top3_push_lex(d, sid[e], d0, d1, d2, i0, i1, i2);
                        }
                    }
                }
            }
            // everything not visited yet is farther than r cells away along some axis
            const float bound = (float)r * h;
            if (i2 >= 0 && d2 < bound * bound - margin) break;
        }
        const long long o = ((long long)p * N + qi) * 3;
        idx[o] = i0; idx[o + 1] = i1; idx[o + 2] = i2;
        const float r0 = __fdiv_rn(1.0f, __fadd_rn(d0, 1e-8f));
        const float r1 = __fdiv_rn(1.0f, __fadd_rn(d1, 1e-8f));
        const float r2 = __fdiv_rn(1.0f, __fadd_rn(d2, 1e-8f));
        const float nrm = __fadd_rn(__fadd_rn(r0, r1), r2);
        if (wout) { wout[o] = __fdiv_rn(r0, nrm); wout[o + 1] = __fdiv_rn(r1, nrm); wout[o + 2] = __fdiv_rn(r2, nrm); }
        if (d2out) { d2out[o] = d0; d2out[o + 1] = d1; d2out[o + 2] = d2; }
    }
}

__global__ void __launch_bounds__(256)
square_distance_kernel(const float *__restrict__ src, const float *__restrict__ dst, int N, int M,
                       float *__restrict__ out)
{
    const int b = blockIdx.z;
    const int i = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    const float *s = src + ((long long)b * N + i) * 3;
    const float *d = dst + ((long long)b * M + j) * 3;
    float sx = s[0], sy = s[1], sz = s[2], dx = d[0], dy = d[1], dz = d[2];
    out[((long long)b * N + i) * M + j] =
        psg_sqdist(sx, sy, sz, psg_sqnorm(sx, sy, sz), dx, dy, dz, psg_sqnorm(dx, dy, dz));
}

}  // namespace

int psg_ball_query_launch(const float *xyz, long long cloud_stride, int nclouds, int P, int N,
                          const float *new_xyz, int S, int nr, const double *radius, const int *nsample,
                          int *out0, int *out1, cudaStream_t st)
{
    if (P <= 0 || N <= 0 || S <= 0 || nr < 1 || nr > 2) return PSG_EINVAL;
    const int warps = S >= 32 ? 32 : (S >= 8 ? 8 : 1);
    dim3 grid((S + warps - 1) / warps, P);
    const size_t smem = 4 * kBallChunk * sizeof(float);
    // pointnet_util.py:102 compares the float32 tensor against radius**2 (a Python double, cast to
    // the tensor dtype by the comparison)
    const float r2a = (float)(radius[0] * radius[0]);
    static PsgDeviceOnce attr_once;
    if (attr_once.need()) {
        if (cudaFuncSetAttribute(ball_query_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
            cudaFuncSetAttribute(ball_query_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return PSG_ECUDA;
        attr_once.mark();
    }
    if (nr == 1) {
        ball_query_kernel<1><<<grid, warps * 32, smem, st>>>(xyz, cloud_stride, nclouds, N, new_xyz, S, r2a, 0.f,
                                                            nsample[0], 0, out0, nullptr);
    } else {
        const float r2b = (float)(radius[1] * radius[1]);
        ball_query_kernel<2><<<grid, warps * 32, smem, st>>>(xyz, cloud_stride, nclouds, N, new_xyz, S, r2a, r2b,
                                                            nsample[0], nsample[1], out0, out1);
    }
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

static int g_nn_grid_mode = 0;      // 0 automatic, 1 never, 2 whenever the coarse cloud fits (tests)
void psg_three_nn_grid_mode(int m) { g_nn_grid_mode = m; }

int psg_three_nn_launch(const float *xyz1, long long stride1, int nclouds1, int P, int N,
                        const float *xyz2, int S, int *idx, float *w, float *d2, cudaStream_t st)
{
    if (P <= 0 || N <= 0 || S < 3) return PSG_EINVAL;
    const bool want_grid = g_nn_grid_mode == 2 ? S <= kNgMaxS
                         : g_nn_grid_mode == 1 ? false : (S >= 256 && S <= kNgMaxS && N >= 1024 && (long long)P * N >= 32768);
    if (want_grid) {
        // many queries against a cloud worth binning: uniform grid (bit-identical results)
        const size_t smem = (size_t)S * 20 + (size_t)(2 * kNgMaxCells + 1) * 4 + 16;
        static PsgDeviceOnce attr_once;
        if (attr_once.need()) {
            if (cudaFuncSetAttribute(three_nn_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kNgMaxS * 20 + (2 * kNgMaxCells + 1) * 4 + 16) != cudaSuccess)
                return PSG_ECUDA;
            attr_once.mark();
        }
        dim3 ggrid((N + kNgQ - 1) / kNgQ, P);
        three_nn_grid_kernel<<<ggrid, 256, smem, st>>>(xyz1, stride1, nclouds1, N, xyz2, S, idx, w, d2);
        PSG_LAUNCH_CHECK();
        return PSG_OK;
    }
    dim3 grid((N + 256 * kNnQ - 1) / (256 * kNnQ), P);
    three_nn_kernel<<<grid, 256, 0, st>>>(xyz1, stride1, nclouds1, N, xyz2, S, idx, w, d2);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

int psg_square_distance_launch(const float *src, const float *dst, int B, int N, int M, float *out,
                               cudaStream_t st)
{
    if (B <= 0 || N <= 0 || M <= 0 || N > 65535 || B > 65535) return PSG_EINVAL;
    dim3 grid((M + 255) / 256, N, B);
    square_distance_kernel<<<grid, 256, 0, st>>>(src, dst, N, M, out);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
