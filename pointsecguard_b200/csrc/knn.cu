// knn.cu -- dense k-nearest-neighbour graph in feature space (SURVEY.md 8f rank 4).
//
// Reference: ResGCN/gcn_lib/dense/torch_edge.py:32-59 -- pairwise_distance(x) = x_square + (-2 x x^T) + x_square^T over
// x [B, N, C], then torch.topk(-distance, k): the k nearest points of every point (itself included, distance 0), nearest
// first.  The reference materialises the [B, N, N] matrix (1 GB per 16 clouds of 4096 points) and sorts it; here no distance
// reaches HBM.  Two kernels, selected by k and C:
//   * k <= 16 and C <= 64: dense_knn_kernel keeps 128 queries per CTA in registers (features + a sorted top-k list each) and
//     streams the cloud through shared memory in tiles.
//   * otherwise (k <= 1024, any C): knn_select_kernel keeps a sorted best-k list and a pending buffer per query in shared
//     memory, streams the cloud in point tiles and channel chunks, and merges the pending candidates into the list with a
//     warp bitonic sort + merge whenever the buffer fills (DESIGN.md section 12 has the measurements behind the split).
// Arithmetic (both kernels, = pairwise_kernel bit for bit): |x|^2 as separately rounded products added left to right, the dot
// product as fmul of channel 0 then an fma chain in ascending channel order, the sum as ((|x_i|^2 + (-2 dot)) + |x_j|^2).
// The reference's sgemm on x x^T accumulates in its own order, so distances agree with it to rounding (measured: 4 of 65 536
// neighbour slots differ at C = 3, each between two candidates whose distances agree to 1e-6 relative).
// Order: strict (distance, index) -- exact ties go to the smaller index (torch.topk leaves them unspecified), NaN distances
// after +inf.  So every output index lies in [0, N) and appears once per row, also on non-finite input.
#include "../../include/psg_b200.h"
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

constexpr int kTile = 64;

// Does a candidate at distance d precede the list entry (e, i)?  Candidates arrive in ascending index, so on equal
// distances the entry (smaller index) stays first.  NaN orders after +inf, and an empty slot (NaN, INT_MAX) after everything.
// On finite distances this is d < e, the comparison the kernel always made.
__device__ __forceinline__ bool precedes(float d, float e, int i)
{
    return d < e || (e != e && (d == d || i == 0x7fffffff));
}

template <int CP, int KMAX>
__global__ void __launch_bounds__(128) dense_knn_kernel(const float *__restrict__ x, int N, int C, int k,
                                                        long long *__restrict__ nn_idx, float *__restrict__ nn_d2)
{
    __shared__ __align__(16) float xs[kTile][CP];
    __shared__ float sq[kTile];
    const int b = blockIdx.y;
    const int i = blockIdx.x * 128 + threadIdx.x;
    const float *xb = x + (size_t)b * N * C;
    float q[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) q[c] = (i < N && c < C) ? xb[(size_t)i * C + c] : 0.f;
    float qs = 0.f;
#pragma unroll
    for (int c = 0; c < CP; ++c) qs = c == 0 ? __fmul_rn(q[0], q[0]) : __fadd_rn(qs, __fmul_rn(q[c], q[c]));
    // empty slots hold (NaN, INT_MAX): every candidate, NaN included, precedes them
    float bd[KMAX];
    int bi[KMAX];
#pragma unroll
    for (int t = 0; t < KMAX; ++t) { bd[t] = __int_as_float(0x7fffffff); bi[t] = 0x7fffffff; }
    for (int j0 = 0; j0 < N; j0 += kTile) {
        __syncthreads();
        for (int e = threadIdx.x; e < kTile * CP; e += 128) {
            const int r = e / CP, c = e - r * CP;
            xs[r][c] = (j0 + r < N && c < C) ? xb[(size_t)(j0 + r) * C + c] : 0.f;
        }
        __syncthreads();
        if (threadIdx.x < kTile) {
            float s = 0.f;
#pragma unroll
            for (int c = 0; c < CP; ++c) s = c == 0 ? __fmul_rn(xs[threadIdx.x][0], xs[threadIdx.x][0]) : __fadd_rn(s, __fmul_rn(xs[threadIdx.x][c], xs[threadIdx.x][c]));
            sq[threadIdx.x] = s;
        }
        __syncthreads();
        const int lim = min(kTile, N - j0);
        for (int r = 0; r < lim; ++r) {
            float dot = __fmul_rn(q[0], xs[r][0]);
#pragma unroll
            for (int c = 1; c < CP; ++c) dot = __fmaf_rn(q[c], xs[r][c], dot);
            const float d = __fadd_rn(__fadd_rn(qs, __fmul_rn(-2.0f, dot)), sq[r]);
            if (precedes(d, bd[KMAX - 1], bi[KMAX - 1])) {
                // sorted insertion; candidates arrive in ascending index, so a strict '<' keeps the smaller index on ties
                const int j = j0 + r;
                bool placed = false;
#pragma unroll
                for (int t = KMAX - 1; t > 0; --t) {
                    if (!placed) {
                        if (precedes(d, bd[t - 1], bi[t - 1])) { bd[t] = bd[t - 1]; bi[t] = bi[t - 1]; }
                        else { bd[t] = d; bi[t] = j; placed = true; }
                    }
                }
                if (!placed) { bd[0] = d; bi[0] = j; }
            }
        }
    }
    if (i < N) {
#pragma unroll
        for (int t = 0; t < KMAX; ++t) {
            if (t < k) {
                nn_idx[((size_t)b * N + i) * k + t] = bi[t];
                if (nn_d2) nn_d2[((size_t)b * N + i) * k + t] = bd[t];
            }
        }
    }
}

template <int CP>
int launch_cp(const float *x, int B, int N, int C, int k, long long *idx, float *d2, cudaStream_t st)
{
    dim3 grid((unsigned)((N + 127) / 128), (unsigned)B);
    dense_knn_kernel<CP, 16><<<grid, 128, 0, st>>>(x, N, C, k, idx, d2);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

// ---- knn_select_kernel: any C, k <= 1024 --------------------------------------------------------------------------------
// A CTA of 8 warps owns Q = 8 * QW queries of one cloud (warp w: queries w*QW ... w*QW + QW-1).  Per point tile of 64
// candidates and per channel chunk of CC channels, the tile and the queries' chunk go to shared memory; lane l accumulates
// the dot products of its warp's QW queries with candidates l and l + 32 (2*QW running dots, kept in registers across
// chunks, one float4 load of a query feeding 8 FMAs).  Each query keeps its best k as sorted 64-bit keys
// (order-preserving bits of the distance << 32 | index: a strict total order, NaN after +inf) in `list`, and a pending buffer
// of kPend keys.  A candidate is appended only if its key precedes the list's k-th entry; when fewer than a tile's worth of
// free slots remain, and once at the end, the owning warp sorts the buffer (bitonic) and merges it into the list in place.
constexpr int kSelWarps = 8, kSelThreads = kSelWarps * 32, kSelTile = 64, kPend = 128, kSelMaxK = 1024;
constexpr unsigned long long kEmpty = ~0ull;      // after every real key: NaN's key is 0xffffffff and indices are < 2^31

__device__ __forceinline__ unsigned dist_key(float d)
{
    const unsigned u = __float_as_uint(d);
    if (d != d) return 0xffffffffu;                // every NaN after +inf (0xff800000)
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // (d is never -0: |x_i|^2 >= +0 and RN gives -0 only for -0 + -0)
}

__device__ __forceinline__ float key_dist(unsigned key)
{
    return __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

// Merge the cnt pending keys P into the sorted list L[0, k) (one warp; P has room for kPend keys; keys are distinct).
__device__ __forceinline__ void merge_pending(unsigned long long *L, int k, unsigned long long *P, int cnt, int lane)
{
    int n2 = 32;
    while (n2 < cnt) n2 <<= 1;
    for (int e = cnt + lane; e < n2; e += 32) P[e] = kEmpty;
    __syncwarp();
    for (int size = 2; size <= n2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int p = lane; p < (n2 >> 1); p += 32) {
                const int a = 2 * p - (p & (stride - 1)), c = a + stride;
                const unsigned long long va = P[a], vc = P[c];
                if ((va > vc) == ((a & size) == 0)) { P[a] = vc; P[c] = va; }
            }
            __syncwarp();
        }
    }
    // final slot of every pending key: its rank in P plus the number of list keys below it (searched before the list moves)
    unsigned long long pv[kPend / 32];
    int pp[kPend / 32];
#pragma unroll
    for (int t = 0; t < kPend / 32; ++t) {
        const int e = lane + 32 * t;
        pp[t] = k;
        pv[t] = 0;
        if (e < cnt) {
            const unsigned long long v = P[e];
            int lo = 0, hi = k;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (L[mid] < v) lo = mid + 1; else hi = mid; }
            pp[t] = e + lo;
            pv[t] = v;
        }
    }
    // list keys below P[0] stay; the others move up by the number of pending keys below them.  Chunks go from the top down
    // and every chunk is read before it is written, so a move (always upwards, to a slot no other key takes) never
    // overwrites a key that has not moved yet.
    int lo0 = 0;
    {
        const unsigned long long v = P[0];
        int hi = k;
        while (lo0 < hi) { const int mid = (lo0 + hi) >> 1; if (L[mid] < v) lo0 = mid + 1; else hi = mid; }
    }
    for (int top = k; top > lo0; top -= 32) {
        const int i = top - 32 + lane;
        const bool act = i >= lo0;
        const unsigned long long v = act ? L[i] : 0ull;
        int r = 0;
        if (act) {
            int hi = n2;
            while (r < hi) { const int mid = (r + hi) >> 1; if (P[mid] < v) r = mid + 1; else hi = mid; }
        }
        __syncwarp();
        if (act && i + r < k) L[i + r] = v;
        __syncwarp();
    }
#pragma unroll
    for (int t = 0; t < kPend / 32; ++t)
        if (pp[t] < k) L[pp[t]] = pv[t];
    __syncwarp();
}

template <int CC, int QW>
__global__ void __launch_bounds__(kSelThreads, 2) knn_select_kernel(const float *__restrict__ x, int N, int C, int k, int nqb,
                                                                 long long *__restrict__ nn_idx, float *__restrict__ nn_d2)
{
    constexpr int S = CC == 4 ? 4 : CC + 4;        // row stride in floats: conflict-free float4 rows across 8 lanes
    constexpr int Q = kSelWarps * QW;
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned long long *list = reinterpret_cast<unsigned long long *>(smem);      // [Q][k]
    unsigned long long *pend = list + (size_t)Q * k;                               // [Q][kPend]
    float *xs = reinterpret_cast<float *>(pend + Q * kPend);                       // [kSelTile][S] candidate chunk
    float *xq = xs + kSelTile * S;                                                 // [Q][S] query chunk
    float *sq = xq + Q * S;                                                        // [kSelTile] |x_j|^2
    float *qs = sq + kSelTile;                                                     // [Q] |x_i|^2
    const int b = blockIdx.x / nqb, i0 = (blockIdx.x - b * nqb) * Q;
    const float *xb = x + (size_t)b * N * C;
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    for (int e = tid; e < Q * k; e += kSelThreads) list[e] = kEmpty;
    if (tid < Q) {
        float s = 0.f;
        if (i0 + tid < N) {
            const float *p = xb + (size_t)(i0 + tid) * C;
            s = __fmul_rn(p[0], p[0]);
            for (int c = 1; c < C; ++c) s = __fadd_rn(s, __fmul_rn(p[c], p[c]));
        }
        qs[tid] = s;
    }
    const int nch = (C + CC - 1) / CC;
    unsigned long long thr[QW];
    int cnt[QW];
#pragma unroll
    for (int t = 0; t < QW; ++t) { thr[t] = kEmpty; cnt[t] = 0; }
    for (int j0 = 0; j0 < N; j0 += kSelTile) {
        float dot[QW][2];
        for (int ch = 0; ch < nch; ++ch) {
            const int c0 = ch * CC;
            __syncthreads();
            for (int e = tid; e < kSelTile * CC; e += kSelThreads) {
                const int r = e / CC, c = e - r * CC;
                xs[r * S + c] = (j0 + r < N && c0 + c < C) ? xb[(size_t)(j0 + r) * C + c0 + c] : 0.f;
            }
            if (nch > 1 || j0 == 0)                // one chunk: the queries stay resident
                for (int e = tid; e < Q * CC; e += kSelThreads) {
                    const int r = e / CC, c = e - r * CC;
                    xq[r * S + c] = (i0 + r < N && c0 + c < C) ? xb[(size_t)(i0 + r) * C + c0 + c] : 0.f;
                }
            __syncthreads();
            const int cl = min(CC, (C - c0 + 3) & ~3);  // channels of this chunk, rounded up to a float4 (zero padded)
            if (tid < kSelTile) {                  // |x_j|^2 continues left to right over the real channels
                float s = ch == 0 ? 0.f : sq[tid];
                for (int c = 0; c < cl && c0 + c < C; ++c) {
                    const float v = xs[tid * S + c];
                    s = c0 + c == 0 ? __fmul_rn(v, v) : __fadd_rn(s, __fmul_rn(v, v));
                }
                sq[tid] = s;
            }
            if (ch == 0) {
                // fma(a, b, -0) rounds a*b once and keeps the sign of a zero product: it is fmul(a, b) bit for bit
#pragma unroll
                for (int t = 0; t < QW; ++t) dot[t][0] = dot[t][1] = -0.f;
            }
            // padded channels are 0 in both operands; fma(0, 0, dot) = dot up to the sign of a zero dot, which the
            // distance cannot see (|x_i|^2 + (-2 dot) with |x_i|^2 >= +0)
#pragma unroll 4
            for (int c = 0; c < cl; c += 4) {
                const float4 ca = *reinterpret_cast<const float4 *>(&xs[lane * S + c]);
                const float4 cb = *reinterpret_cast<const float4 *>(&xs[(lane + 32) * S + c]);
#pragma unroll
                for (int t = 0; t < QW; ++t) {
                    const float4 q = *reinterpret_cast<const float4 *>(&xq[(w * QW + t) * S + c]);
                    dot[t][0] = __fmaf_rn(q.x, ca.x, dot[t][0]);
                    dot[t][1] = __fmaf_rn(q.x, cb.x, dot[t][1]);
                    dot[t][0] = __fmaf_rn(q.y, ca.y, dot[t][0]);
                    dot[t][1] = __fmaf_rn(q.y, cb.y, dot[t][1]);
                    dot[t][0] = __fmaf_rn(q.z, ca.z, dot[t][0]);
                    dot[t][1] = __fmaf_rn(q.z, cb.z, dot[t][1]);
                    dot[t][0] = __fmaf_rn(q.w, ca.w, dot[t][0]);
                    dot[t][1] = __fmaf_rn(q.w, cb.w, dot[t][1]);
                }
            }
        }
        __syncthreads();                           // sq complete
        const float sa = sq[lane], sb = sq[lane + 32];
        const unsigned lt = (1u << lane) - 1u;
#pragma unroll
        for (int t = 0; t < QW; ++t) {
            const int ql = w * QW + t;
            const bool qv = i0 + ql < N;
            const float q2 = qs[ql];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = j0 + lane + 32 * h;
                const float d = __fadd_rn(__fadd_rn(q2, __fmul_rn(-2.0f, dot[t][h])), h ? sb : sa);
                const unsigned long long key = ((unsigned long long)dist_key(d) << 32) | (unsigned)j;
                const bool pass = qv && j < N && key < thr[t];
                const unsigned m = __ballot_sync(0xffffffffu, pass);
                if (pass) pend[ql * kPend + cnt[t] + __popc(m & lt)] = key;
                cnt[t] += __popc(m);
            }
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < QW; ++t) {
            if (cnt[t] > kPend - kSelTile) {
                const int ql = w * QW + t;
                merge_pending(list + (size_t)ql * k, k, pend + ql * kPend, cnt[t], lane);
                cnt[t] = 0;
                thr[t] = list[(size_t)ql * k + k - 1];
            }
        }
    }
    __syncwarp();
#pragma unroll
    for (int t = 0; t < QW; ++t) {
        const int ql = w * QW + t, i = i0 + ql;
        if (cnt[t] > 0) merge_pending(list + (size_t)ql * k, k, pend + ql * kPend, cnt[t], lane);
        if (i < N) {
            const unsigned long long *Lq = list + (size_t)ql * k;
            for (int e = lane; e < k; e += 32) {
                const unsigned long long v = Lq[e];
                nn_idx[((size_t)b * N + i) * k + e] = (long long)(unsigned)(v & 0xffffffffu);
                if (nn_d2) nn_d2[((size_t)b * N + i) * k + e] = key_dist((unsigned)(v >> 32));
            }
        }
    }
}

template <int CC>
size_t select_smem(int QW, int k)
{
    const int S = CC == 4 ? 4 : CC + 4, Q = kSelWarps * QW;
    return (size_t)Q * (k + kPend) * 8 + (size_t)(kSelTile * S + Q * S + kSelTile + Q) * 4;
}

template <int CC, int QW>
int launch_select_qw(const float *x, int B, int N, int C, int k, long long *idx, float *d2, cudaStream_t st)
{
    const size_t smem = select_smem<CC>(QW, k);
    if (cudaFuncSetAttribute(knn_select_kernel<CC, QW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return PSG_ECUDA;
    const int nqb = (N + kSelWarps * QW - 1) / (kSelWarps * QW);
    if ((long long)nqb * B > 0x7fffffffLL) return PSG_EUNSUPPORTED;
    knn_select_kernel<CC, QW><<<(unsigned)(nqb * B), kSelThreads, smem, st>>>(x, N, C, k, nqb, idx, d2);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

// Queries per warp: the most that still let two CTAs share an SM (16 warps; 4 queries per warp is the most that stays within
// the 128 registers of that occupancy without spilling).  At k = 1024 one query per warp takes 94 KB.
template <int CC>
int launch_select(const float *x, int B, int N, int C, int k, long long *idx, float *d2, cudaStream_t st)
{
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return PSG_ECUDA;
    const size_t cap = (size_t)optin / 2 - 1024;  // the 1 KB the driver reserves per CTA
    if (select_smem<CC>(4, k) <= cap) return launch_select_qw<CC, 4>(x, B, N, C, k, idx, d2, st);
    if (select_smem<CC>(2, k) <= cap) return launch_select_qw<CC, 2>(x, B, N, C, k, idx, d2, st);
    if (select_smem<CC>(1, k) <= cap) return launch_select_qw<CC, 1>(x, B, N, C, k, idx, d2, st);
    return PSG_EUNSUPPORTED;
}

// full matrix, for the API function pairwise_distance (tests / small clouds)
__global__ void pairwise_kernel(const float *__restrict__ x, int N, int C, float *__restrict__ out)
{
    const int b = blockIdx.z;
    const int i = blockIdx.y * blockDim.y + threadIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || j >= N) return;
    const float *xi = x + ((size_t)b * N + i) * C, *xj = x + ((size_t)b * N + j) * C;
    float si = __fmul_rn(xi[0], xi[0]), sj = __fmul_rn(xj[0], xj[0]), dot = __fmul_rn(xi[0], xj[0]);
    for (int c = 1; c < C; ++c) {
        si = __fadd_rn(si, __fmul_rn(xi[c], xi[c]));
        sj = __fadd_rn(sj, __fmul_rn(xj[c], xj[c]));
        dot = __fmaf_rn(xi[c], xj[c], dot);
    }
    out[((size_t)b * N + i) * N + j] = __fadd_rn(__fadd_rn(si, __fmul_rn(-2.0f, dot)), sj);
}

}  // namespace

extern "C" int psg_dense_knn(const float *x, int B, int N, int C, int k, int64_t *nn_idx, float *nn_d2, psg_stream_t stream)
{
    if (!x || !nn_idx || B <= 0 || N <= 0 || C <= 0 || k <= 0 || k > kSelMaxK || k > N) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    long long *idx = reinterpret_cast<long long *>(nn_idx);
    // k <= 16 and C <= 64: the register kernel.  Above that the list kernel is faster: measured on a B200 at 1000 W, 16 x 4096
    // points, the register kernel took 11.0 ms (C = 3) / 13.0 ms (C = 64) at k = 32, the list kernel 2.6 / 4.8 ms at k = 33
    // (DESIGN.md section 12, profiles/knn_bench*.json).
    if (k > 16 || C > 64) {
        if (C <= 4) return launch_select<4>(x, B, N, C, k, idx, nn_d2, st);
        if (C <= 16) return launch_select<16>(x, B, N, C, k, idx, nn_d2, st);
        return launch_select<64>(x, B, N, C, k, idx, nn_d2, st);
    }
    if (C <= 4) return launch_cp<4>(x, B, N, C, k, idx, nn_d2, st);
    if (C <= 8) return launch_cp<8>(x, B, N, C, k, idx, nn_d2, st);
    if (C <= 16) return launch_cp<16>(x, B, N, C, k, idx, nn_d2, st);
    if (C <= 32) return launch_cp<32>(x, B, N, C, k, idx, nn_d2, st);
    return launch_cp<64>(x, B, N, C, k, idx, nn_d2, st);
}

extern "C" int psg_pairwise_distance(const float *x, int B, int N, int C, float *out, psg_stream_t stream)
{
    if (!x || !out || B <= 0 || N <= 0 || C <= 0) return PSG_EINVAL;
    dim3 block(32, 8), grid((unsigned)((N + 31) / 32), (unsigned)((N + 7) / 8), (unsigned)B);
    pairwise_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(x, N, C, out);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
