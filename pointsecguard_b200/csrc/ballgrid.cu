// ballgrid.cu -- ball query over a uniform grid (large clouds).
//
// Reference semantics (PointNet/models/pointnet_util.py:87-107): for each centroid the indices of the
// points with d2 <= r^2 in ASCENDING INDEX order, the first `nsample` of them, unfilled slots = the
// first hit (N when there is none); d2 is the expansion-form square_distance(new_xyz, xyz).
//
// The brute-force kernel (neighbors.cu) tests every point for every centroid: 4096 x 1024 distance
// evaluations per SA1 cloud, ~5 hits each -- the largest item of the per-step geometry cost.  Here the
// cloud is binned once into cells of edge >= 1.01 r (+1e-4), a centroid only tests the points of its
// 27 neighbouring cells (the membership test is per pair, so using the same oracle-exact formula on a
// superset of the hits gives bit-identical membership), and the hits -- found in cell order -- are
// emitted smallest index first.  A centroid with more hits than the per-warp list holds falls back to
// the exhaustive scan.
//
// The superset holds only while the formula's rounding error stays below the cell margin cell^2 - r^2,
// and that error grows with the coordinates, not with r.  With u = 2^-24, Q = |q|^2 (centroid), P = |p|^2
// (point) and M = max |p|^2 over the cloud: psg_sqdist's dot (one multiply, two FMAs) is within 3u |q||p|,
// |q|^2 and |p|^2 (three roundings each) within 3u Q and 3u P, and the two rounded adds add u (2Q + P)
// and u d2, so the computed d2 is within 8u (Q + P) + u d2 of |q - p|^2.  Cell indices are rounded too
// ((x - min) * inv_cell: three roundings, plus the clamp of the last cell), so a point outside the 27
// cells may lie up to 3u (|q| + 5 sqrt(M)) nearer than one cell edge along the separating axis; squared,
// that costs at most 3u Q + 15u M + 18u cell^2.  Such a point cannot be a hit when
// 23u (Q + M) + 19u cell^2 < cell^2 - r^2.  ball_grid_kernel requires the stronger
//     2^-19 (Q + M + cell^2) < cell^2 - r^2          (2^-19 = 32u: 1.4x the bound, covering the test's own rounding)
// and sends every other centroid straight to the exhaustive scan.  At r = 0.1 (cell 0.1011) that admits
// Q + M < 116 m^2, and even an ungrown cell at r = 0.05 (0.0506) admits Q + M < 31 m^2, so a 1 x 1 x 3 m block
// at the origin (Q + M <= 19) keeps the grid for every centroid; a cloud tens of metres from the origin scans
// unless its cell grew large (a scene-sized slab).  A cloud with a non-finite coordinate, or whose M
// overflows, is not binned at all and every centroid scans, so a NaN distance counts as a hit exactly as
// the reference counts it (!(d > r^2)).
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

constexpr int kMaxCells = 16384;
constexpr int kCap = 96;            // hits kept per warp and radius before falling back (3 per lane)
constexpr int kWarps = 8;

struct GridHdr {
    float minx, miny, minz, inv_cell;
    int gx, gy, gz, ncells;
    float cell, m2;         // cell edge, max |p|^2 of the cloud
    int finite;             // 0: a coordinate or an |p|^2 is not finite -- the cloud was not binned, every centroid scans
};

__host__ __device__ inline size_t grid_bytes_per_cloud(int N)
{
    // header | cell_start[kMaxCells + 1] | cursor[kMaxCells] | sorted xyzn float4[N] | sorted idx[N]
    size_t b = 256 + (size_t)(2 * kMaxCells + 1) * 4;
    b = (b + 15) & ~(size_t)15;
    b += (size_t)N * 16 + (size_t)N * 4;
    return (b + 255) & ~(size_t)255;
}
__device__ inline GridHdr *g_hdr(unsigned char *ws) { return reinterpret_cast<GridHdr *>(ws); }
__device__ inline int *g_start(unsigned char *ws) { return reinterpret_cast<int *>(ws + 256); }
__device__ inline int *g_cursor(unsigned char *ws) { return g_start(ws) + kMaxCells + 1; }
__device__ inline float4 *g_pts(unsigned char *ws)
{
    size_t b = 256 + (size_t)(2 * kMaxCells + 1) * 4;
    b = (b + 15) & ~(size_t)15;
    return reinterpret_cast<float4 *>(ws + b);
}
__device__ inline int *g_idx(unsigned char *ws, int N) { return reinterpret_cast<int *>(g_pts(ws) + N); }

__device__ __forceinline__ int cell_of(const GridHdr &h, float x, float y, float z)
{
    int cx = (int)floorf((x - h.minx) * h.inv_cell), cy = (int)floorf((y - h.miny) * h.inv_cell),
        cz = (int)floorf((z - h.minz) * h.inv_cell);
    cx = min(max(cx, 0), h.gx - 1); cy = min(max(cy, 0), h.gy - 1); cz = min(max(cz, 0), h.gz - 1);
    return (cz * h.gy + cy) * h.gx + cx;
}

// one CTA per cloud: bounding box -> cell size -> counting sort of the points by cell
__global__ void __launch_bounds__(1024) grid_build_kernel(const float *__restrict__ xyz, long long cloud_stride, int N,
                                                          float rmax, unsigned char *__restrict__ ws_all, size_t ws_stride)
{
    __shared__ float red[7][32];
    __shared__ GridHdr hdr;
    __shared__ int wsum[32];
    __shared__ int carry_s;
    const float *cloud = xyz + (long long)blockIdx.x * cloud_stride;
    unsigned char *ws = ws_all + (size_t)blockIdx.x * ws_stride;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY}, m2 = 0.f;
    bool fin = true;
    for (int i = t; i < N; i += blockDim.x) {
        const float x = cloud[3 * i], y = cloud[3 * i + 1], z = cloud[3 * i + 2];
        lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
        hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
        m2 = fmaxf(m2, psg_sqnorm(x, y, z));
        fin = fin && isfinite(x) && isfinite(y) && isfinite(z);     // fminf / fmaxf skip a NaN: count it here
    }
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if (lane == 0) { red[a][warp] = lo[a]; red[3 + a][warp] = hi[a]; }
    }
    for (int o = 16; o > 0; o >>= 1) m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, o));
    if (lane == 0) red[6][warp] = m2;
    const bool all_finite = __syncthreads_and(fin);
    if (t == 0) {
        float l[3], h[3], mm = red[6][0];
        for (int a = 0; a < 3; ++a) {
            l[a] = red[a][0]; h[a] = red[3 + a][0];
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { l[a] = fminf(l[a], red[a][w]); h[a] = fmaxf(h[a], red[3 + a][w]); }
        }
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mm = fmaxf(mm, red[6][w]);
        // finite coordinates with a finite max |p|^2 bound every extent below 4e19: the cell counts below stay finite
        hdr.finite = all_finite && mm < INFINITY;
        float cell = rmax * 1.01f + 1e-4f, fx = 1.f, fy = 1.f, fz = 1.f;
        if (hdr.finite) {
            for (;;) {                           // counted in float: an extent of 2^31 cells must not wrap an int
                fx = floorf((h[0] - l[0]) / cell) + 1.f; fy = floorf((h[1] - l[1]) / cell) + 1.f;
                fz = floorf((h[2] - l[2]) / cell) + 1.f;
                if ((double)fx * fy * fz <= kMaxCells) break;
                cell *= 1.26f;                   // ~ halves the cell count
            }
        }
        hdr.minx = l[0]; hdr.miny = l[1]; hdr.minz = l[2]; hdr.inv_cell = 1.0f / cell;
        hdr.gx = (int)fx; hdr.gy = (int)fy; hdr.gz = (int)fz; hdr.ncells = hdr.gx * hdr.gy * hdr.gz;
        hdr.cell = cell; hdr.m2 = mm;
        *g_hdr(ws) = hdr;
        carry_s = 0;
    }
    __syncthreads();
    if (!hdr.finite) return;                     // not binned: ball_grid_kernel scans every centroid of this cloud
    int *start = g_start(ws), *cursor = g_cursor(ws);
    const int nc = hdr.ncells;
    for (int c = t; c <= nc; c += blockDim.x) start[c] = 0;
    for (int c = t; c < nc; c += blockDim.x) cursor[c] = 0;
    __syncthreads();
    for (int i = t; i < N; i += blockDim.x) atomicAdd(&start[cell_of(hdr, cloud[3 * i], cloud[3 * i + 1], cloud[3 * i + 2])], 1);
    __syncthreads();
    // exclusive scan of start[0..nc) in place, start[nc] = N
    for (int base = 0; base < nc; base += blockDim.x) {
        const int c = base + t;
        const int v = c < nc ? start[c] : 0;
        int x = v;
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int s = wsum[lane];
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
            wsum[lane] = s;
        }
        __syncthreads();
        const int incl = x + (warp ? wsum[warp - 1] : 0) + carry_s;
        if (c < nc) start[c] = incl - v;
        __syncthreads();
        if (t == (int)blockDim.x - 1) carry_s = incl;
        __syncthreads();
    }
    if (t == 0) start[nc] = N;
    __syncthreads();
    float4 *pts = g_pts(ws);
    int *sidx = g_idx(ws, N);
    for (int i = t; i < N; i += blockDim.x) {
        const float x = cloud[3 * i], y = cloud[3 * i + 1], z = cloud[3 * i + 2];
        const int c = cell_of(hdr, x, y, z);
        const int pos = start[c] + atomicAdd(&cursor[c], 1);     // order inside a cell is irrelevant: hits are re-ordered
        pts[pos] = make_float4(x, y, z, psg_sqnorm(x, y, z));
        sidx[pos] = i;
    }
}

// append the ids of the lanes set in `m` (warp-uniform) to the hit list: slot p lives in lane p % 32, register p / 32
__device__ __forceinline__ void push_hits(unsigned m, int id, int lane, int &cnt, int &h0, int &h1, int &h2)
{
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const int v = __shfl_sync(0xffffffffu, id, src);
        if (cnt < kCap && (cnt & 31) == lane) { if (cnt < 32) h0 = v; else if (cnt < 64) h1 = v; else h2 = v; }
        ++cnt;
    }
}

// emit the first K of `cnt` hit indices (3 per lane in h[]) in ascending order, pad with the smallest
__device__ __forceinline__ void emit_sorted(int h0, int h1, int h2, int cnt, int K, int N, int *out, int lane)
{
    const int kmax = 0x7fffffff;
    int first = N;
    const int n = min(cnt, K);
    for (int k = 0; k < n; ++k) {
        const int m = __reduce_min_sync(0xffffffffu, min(h0, min(h1, h2)));
        if (k == 0) first = m;
        if (lane == 0) out[k] = m;
        if (h0 == m) h0 = kmax; else if (h1 == m) h1 = kmax; else if (h2 == m) h2 = kmax;
    }
    for (int k = n + lane; k < K; k += 32) out[k] = first;
}

template <int NR>
__global__ void __launch_bounds__(kWarps * 32)
ball_grid_kernel(const unsigned char *__restrict__ ws_all, size_t ws_stride, const float *__restrict__ xyz, long long cloud_stride,
                 int nclouds, int N, const float *__restrict__ new_xyz, int S, float r2a, float r2b, int Ka, int Kb,
                 int *__restrict__ outa, int *__restrict__ outb)
{
    const int p = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * kWarps + warp;
    if (s >= S) return;
    const int cloud_id = p % nclouds;
    unsigned char *ws = const_cast<unsigned char *>(ws_all) + (size_t)cloud_id * ws_stride;
    const GridHdr h = *g_hdr(ws);
    const int *start = g_start(ws);
    const float4 *pts = g_pts(ws);
    const int *sidx = g_idx(ws, N);
    const float *q = new_xyz + ((long long)p * S + s) * 3;
    const float qx = q[0], qy = q[1], qz = q[2], qn = psg_sqnorm(qx, qy, qz);
    int *oa = outa + ((long long)p * S + s) * Ka;
    int *ob = NR == 2 ? outb + ((long long)p * S + s) * Kb : nullptr;

    const int kmax = 0x7fffffff;
    int a0 = kmax, a1 = kmax, a2 = kmax, b0 = kmax, b1 = kmax, b2 = kmax;   // hit lists, 3 slots per lane
    int cnta = 0, cntb = 0;
    // the margin rule of the file comment: the 27 cells hold every hit only when the rounding error of the distance
    // formula is proven to stay inside cell^2 - r^2 (false for a NaN centroid and for a cloud that was not binned)
    const float r2max = NR == 2 ? fmaxf(r2a, r2b) : r2a;
    bool scan = !h.finite || !(0x1p-19f * ((qn + h.m2) + h.cell * h.cell) < h.cell * h.cell - r2max);
    int cx = (int)floorf((qx - h.minx) * h.inv_cell), cy = (int)floorf((qy - h.miny) * h.inv_cell),
        cz = (int)floorf((qz - h.minz) * h.inv_cell);
    for (int dz = -1; dz <= 1 && !scan; ++dz) {
        const int z = cz + dz;
        if (z < 0 || z >= h.gz) continue;
        for (int dy = -1; dy <= 1 && !scan; ++dy) {
            const int y = cy + dy;
            if (y < 0 || y >= h.gy) continue;
            // the three x-neighbours are consecutive cells: one contiguous range of sorted points
            const int x0 = max(cx - 1, 0), x1 = min(cx + 1, h.gx - 1);
            if (x0 > x1) continue;
            const int base = (z * h.gy + y) * h.gx;
            const int lo = start[base + x0], hi = start[base + x1 + 1];
            for (int j0 = lo; j0 < hi; j0 += 32) {
                const int j = j0 + lane;
                bool ha = false, hb = false;
                int id = kmax;
                if (j < hi) {
                    const float4 pt = pts[j];
                    const float d = psg_sqdist(qx, qy, qz, qn, pt.x, pt.y, pt.z, pt.w);
                    ha = !(d > r2a);
                    if (NR == 2) hb = !(d > r2b);
                    id = sidx[j];
                }
                push_hits(__ballot_sync(0xffffffffu, ha), id, lane, cnta, a0, a1, a2);
                if (NR == 2) push_hits(__ballot_sync(0xffffffffu, hb), id, lane, cntb, b0, b1, b2);
                if (cnta > kCap || cntb > kCap) { scan = true; break; }
            }
        }
    }
    if (!scan) {
        emit_sorted(a0, a1, a2, cnta, Ka, N, oa, lane);
        if (NR == 2) emit_sorted(b0, b1, b2, cntb, Kb, N, ob, lane);
        return;
    }
    // ---- fallback: exhaustive scan in index order (dense neighbourhoods; centroids outside the margin rule) ----
    const float *cloud = xyz + (long long)cloud_id * cloud_stride;
    cnta = cntb = 0;
    int firsta = -1, firstb = -1;
    for (int b = 0; b < N; b += 32) {
        const int i = b + lane;
        bool ha = false, hb = false;
        if (i < N) {
            const float x = cloud[3 * i], y = cloud[3 * i + 1], z = cloud[3 * i + 2];
            const float d = psg_sqdist(qx, qy, qz, qn, x, y, z, psg_sqnorm(x, y, z));
            ha = !(d > r2a);
            if (NR == 2) hb = !(d > r2b);
        }
        const unsigned ma = __ballot_sync(0xffffffffu, ha && cnta < Ka);
        if (ma) {
            if (firsta < 0) firsta = b + __ffs(ma) - 1;
            const int pos = cnta + __popc(ma & ((1u << lane) - 1u));
            if (ha && pos < Ka) oa[pos] = i;
            cnta = min(Ka, cnta + __popc(ma));
        }
        if (NR == 2) {
            const unsigned mb = __ballot_sync(0xffffffffu, hb && cntb < Kb);
            if (mb) {
                if (firstb < 0) firstb = b + __ffs(mb) - 1;
                const int pos = cntb + __popc(mb & ((1u << lane) - 1u));
                if (hb && pos < Kb) ob[pos] = i;
                cntb = min(Kb, cntb + __popc(mb));
            }
        }
        if (cnta >= Ka && (NR == 1 || cntb >= Kb)) break;
    }
    const int fa = firsta < 0 ? N : firsta;
    for (int k = cnta + lane; k < Ka; k += 32) oa[k] = fa;
    if (NR == 2) {
        const int fb = firstb < 0 ? N : firstb;
        for (int k = cntb + lane; k < Kb; k += 32) ob[k] = fb;
    }
}

}  // namespace

size_t psg_ballgrid_workspace_bytes(int nclouds, int N) { return (size_t)nclouds * grid_bytes_per_cloud(N); }

int psg_ballgrid_build(const float *xyz, long long cloud_stride, int nclouds, int N, double rmax, void *ws, cudaStream_t st)
{
    if (!xyz || !ws || nclouds <= 0 || N <= 0 || !(rmax > 0.0)) return PSG_EINVAL;
    grid_build_kernel<<<nclouds, 1024, 0, st>>>(xyz, cloud_stride, N, (float)rmax, (unsigned char *)ws, grid_bytes_per_cloud(N));
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

int psg_ballgrid_query(const void *ws, const float *xyz, long long cloud_stride, int nclouds, int P, int N, const float *new_xyz,
                       int S, int nr, const double *radius, const int *nsample, int *out0, int *out1, cudaStream_t st)
{
    if (P <= 0 || N <= 0 || S <= 0 || nr < 1 || nr > 2) return PSG_EINVAL;
    dim3 grid((S + kWarps - 1) / kWarps, P);
    const float r2a = (float)(radius[0] * radius[0]);
    if (nr == 1) {
        ball_grid_kernel<1><<<grid, kWarps * 32, 0, st>>>((const unsigned char *)ws, grid_bytes_per_cloud(N), xyz, cloud_stride,
                                                          nclouds, N, new_xyz, S, r2a, 0.f, nsample[0], 0, out0, nullptr);
    } else {
        const float r2b = (float)(radius[1] * radius[1]);
        ball_grid_kernel<2><<<grid, kWarps * 32, 0, st>>>((const unsigned char *)ws, grid_bytes_per_cloud(N), xyz, cloud_stride,
                                                          nclouds, N, new_xyz, S, r2a, r2b, nsample[0], nsample[1], out0, out1);
    }
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
