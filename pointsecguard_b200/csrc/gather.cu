// gather.cu -- data movement around the shared MLPs, all on T-layout tensors (psg_common.cuh):
//   * pack / unpack between the API's channel-first [B,C,N] tensors and T-layout
//   * SA grouping: gather neighbours, centre xyz, concat      (pointnet_util.py:126-137, :245-255)
//   * neighbourhood max-pool + argmax and its backward         (pointnet_util.py:205, :262)
//   * 3-NN inverse-distance interpolation                      (pointnet_util.py:305-308)
//   * deterministic backward of both gathers: a source-sorted CSR built once per geometry and an
//     ordered segmented sum -- no floating-point atomics anywhere (autograd's index_put_(accumulate)
//     uses atomics on a GPU and is run-to-run nondeterministic)
//   * row-major index_points for the public op                 (pointnet_util.py:43-60)
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

// ---- API <-> T-layout ------------------------------------------------------------------------
// x [B,C,N] with arbitrary strides -> T [B*N][Cpad] (zero padded) and optionally xyz [B][N][3]
__global__ void pack_cf_kernel(const float *__restrict__ x, long long sb, long long sc, long long sn,
                               int B, int C, int N, TView out, int cpad, float *__restrict__ xyz)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= (long long)B * N) return;
    const int b = (int)(row / N), n = (int)(row % N);
    const float *src = x + b * sb + n * sn;
    for (int c = 0; c < cpad / 4; ++c) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int ch = 4 * c + j;
            v[j] = ch < C ? src[ch * sc] : 0.f;
        }
        tv_st(out, row, c, make_float4(v[0], v[1], v[2], v[3]));
    }
    if (xyz) {
        xyz[row * 3 + 0] = src[0];
        xyz[row * 3 + 1] = src[sc];
        xyz[row * 3 + 2] = src[2 * sc];
    }
}

// T [B*N][>=C] -> y [B,C,N] contiguous (optionally accumulate)
__global__ void unpack_cf_kernel(TView in, int B, int C, int N, float *__restrict__ y, int accumulate)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= (long long)B * N) return;
    const int b = (int)(row / N), n = (int)(row % N);
    for (int c = 0; c < (C + 3) / 4; ++c) {
        float4 v = tv_ld(in, row, c);
        float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int ch = 4 * c + j;
            if (ch < C) {
                float *o = y + ((long long)b * C + ch) * N + n;
                *o = accumulate ? *o + a[j] : a[j];
            }
        }
    }
}

// row-major [rows][C] -> T-layout (zero padded) and back
__global__ void pack_rm_kernel(const float *__restrict__ x, long long rows, int C, TView out, int cpad)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int nch = cpad / 4;
    const long long row = t % rows;         // consecutive threads -> consecutive rows of one chunk
    const int c = (int)(t / rows);
    if (c >= nch) return;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { int ch = 4 * c + j; v[j] = ch < C ? x[row * C + ch] : 0.f; }
    tv_st(out, row, c, make_float4(v[0], v[1], v[2], v[3]));
}
__global__ void unpack_rm_kernel(TView in, long long rows, int C, float *__restrict__ y)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int nch = (C + 3) / 4;
    const long long row = t % rows;
    const int c = (int)(t / rows);
    if (c >= nch) return;
    float4 v = tv_ld(in, row, c);
    float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { int ch = 4 * c + j; if (ch < C) y[row * C + ch] = a[j]; }
}

// ---- SA grouping -----------------------------------------------------------------------------
// out row (p,s,k) = [ feats[src] (D) | xyz[src] - new_xyz[p,s] (3) | 0 ... ]
__global__ void group_kernel(TView feats, int D, const float *__restrict__ xyz, long long cloud_stride,
                             int nclouds, int Nsrc, const float *__restrict__ new_xyz,
                             const int *__restrict__ idx, int P, int S, int K, TView out, int cpad)
{
    const long long rows = (long long)P * S * K;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = t % rows;
    const int c = (int)(t / rows);
    if (c >= cpad / 4) return;
    const int p = (int)(row / ((long long)S * K));
    const long long ps = row / K;                         // p*S + s
    const int src = idx[row];
    const int cloud = p % nclouds;
    // feats rows are per problem when the source level is itself per problem (nclouds == P) and
    // shared across iterations for level 0 (nclouds == B)
    const long long srow = (long long)cloud * Nsrc + src;
    float4 v;
    if (4 * c + 3 < D) {
        v = tv_ld(feats, srow, c);
    } else {
        float a[4];
        float4 f = (4 * c < D) ? tv_ld(feats, srow, c) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float fa[4] = {f.x, f.y, f.z, f.w};
        const float *sp = xyz + (long long)cloud * cloud_stride + (long long)src * 3;
        const float *cp = new_xyz + ps * 3;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int ch = 4 * c + j;
            if (ch < D) a[j] = fa[j];
            else if (ch < D + 3) a[j] = __fsub_rn(sp[ch - D], cp[ch - D]);
            else a[j] = 0.f;
        }
        v = make_float4(a[0], a[1], a[2], a[3]);
    }
    tv_st(out, row, c, v);
}

// ---- neighbourhood max-pool ------------------------------------------------------------------
// in rows (g,k), k < K in {16,32}; out[g][col0 + c] = max_k; arg[g][c] = first k attaining it.
// One warp handles 32/K groups; lane = (group-in-warp, k); values are post-ReLU (>= 0) so their
// bit patterns order like unsigned integers and one REDUX gives the max.
template <int K>
__global__ void __launch_bounds__(256)
maxpool_kernel(TView in, long long groups, int C, TView out, unsigned char *__restrict__ arg)
{
    constexpr int GPW = 32 / K;
    const int nch = C / 4;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (group set, chunk)
    const int lane = threadIdx.x & 31;
    const long long gs = wid / nch;
    const int c = (int)(wid % nch);
    const long long g0 = gs * GPW;
    if (g0 >= groups) return;
    const int sub = lane / K, k = lane % K;
    const long long g = g0 + sub;
    const unsigned mask = (K == 32) ? 0xffffffffu : (0xffffu << (16 * sub));
    const bool valid = g < groups;
    const long long row = (valid ? g : g0) * K + k;
    float4 v = tv_ld(in, row, c);
    unsigned b[4] = {__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w)};
    float m[4]; int a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        unsigned mx = __reduce_max_sync(mask, b[j]);
        int cand = (b[j] == mx) ? k : 64;
        a[j] = __reduce_min_sync(mask, cand);
        m[j] = __uint_as_float(mx);
    }
    if (k == 0 && valid) {
        tv_st(out, g, c, make_float4(m[0], m[1], m[2], m[3]));
        *reinterpret_cast<uchar4 *>(arg + g * C + 4 * c) = make_uchar4(a[0], a[1], a[2], a[3]);
    }
}

// dY[(g,k)][c] = (k == arg[g][c] && out[g][c] > 0) ? dOut[g][col0 + c] : 0
template <int K>
__global__ void __launch_bounds__(256)
maxpool_bwd_kernel(TView dout, TView outv, const unsigned char *__restrict__ arg, long long groups, int C,
                   TView dy)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long rows = groups * K;
    const long long row = t % rows;
    const int c = (int)(t / rows);
    if (c >= C / 4) return;
    const long long g = row / K;
    const int k = (int)(row % K);
    float4 d = tv_ld(dout, g, c);
    float4 o = tv_ld(outv, g, c);
    uchar4 a = *reinterpret_cast<const uchar4 *>(arg + g * C + 4 * c);
    float4 r;
    r.x = (a.x == k && o.x > 0.f) ? d.x : 0.f;
    r.y = (a.y == k && o.y > 0.f) ? d.y : 0.f;
    r.z = (a.z == k && o.z > 0.f) ? d.z : 0.f;
    r.w = (a.w == k && o.w > 0.f) ? d.w : 0.f;
    tv_st(dy, row, c, r);
}

// ---- 3-NN interpolation ----------------------------------------------------------------------
// out[p*N+n][c] = (f[i0]*w0 + f[i1]*w1) + f[i2]*w2, products rounded separately as torch does
__global__ void interp_kernel(TView feats, int S, const int *__restrict__ idx, const float *__restrict__ w,
                              long long rows, int N, int nch, TView out)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");          // launched with programmatic stream serialization
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = t % rows;
    const int c = (int)(t / rows);
    if (c >= nch) return;
    const long long p = row / N;
    const int *ii = idx + row * 3;
    const float *ww = w + row * 3;
    const long long base = p * S;
    float4 a = tv_ld(feats, base + ii[0], c), b = tv_ld(feats, base + ii[1], c), d = tv_ld(feats, base + ii[2], c);
    const float w0 = ww[0], w1 = ww[1], w2 = ww[2];
    float4 r;
    r.x = __fadd_rn(__fadd_rn(__fmul_rn(a.x, w0), __fmul_rn(b.x, w1)), __fmul_rn(d.x, w2));
    r.y = __fadd_rn(__fadd_rn(__fmul_rn(a.y, w0), __fmul_rn(b.y, w1)), __fmul_rn(d.y, w2));
    r.z = __fadd_rn(__fadd_rn(__fmul_rn(a.z, w0), __fmul_rn(b.z, w1)), __fmul_rn(d.z, w2));
    r.w = __fadd_rn(__fadd_rn(__fmul_rn(a.w, w0), __fmul_rn(b.w, w1)), __fmul_rn(d.w, w2));
    tv_st(out, row, c, r);
}

// ---- CSR by source (built once per geometry) ------------------------------------------------------
// `grp` > 0: keys are ball-query rows of grp slots; a slot k > 0 holding the group's first hit is
// padding (pointnet_util.py:104-106).  Padded rows are exact copies of the first row, the max-pool
// routes the gradient to the first of equal rows, so their gradient rows are exactly zero: they are
// left out of the CSR (6x fewer entries at SA1 densities, and no 200-entry buckets).
__device__ __forceinline__ bool csr_is_pad(const int *__restrict__ keys, long long t, int slot, int key, int grp)
{
    if (grp <= 0) return false;
    const int k = slot % grp;
    return k > 0 && key == keys[t - k];
}
__global__ void csr_count_kernel(const int *__restrict__ keys, long long total, int M, int R, int grp, int *__restrict__ cnt)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const long long p = t / M;
    const int key = keys[t];
    if (key >= 0 && key < R && !csr_is_pad(keys, t, (int)(t % M), key, grp)) atomicAdd(cnt + p * (R + 1) + key, 1);
}
// exclusive scan of cnt[p][0..R) in place -> offsets[p][0..R]; one CTA per problem
__global__ void __launch_bounds__(1024) csr_scan_kernel(int *__restrict__ cnt, int R)
{
    __shared__ int wsum[32];
    __shared__ int carry_s;
    int *row = cnt + (long long)blockIdx.x * (R + 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < R; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < R ? row[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int s = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
            wsum[lane] = s;
        }
        __syncthreads();
        const int carry = carry_s;
        const int incl = x + (warp ? wsum[warp - 1] : 0) + carry;
        if (i < R) row[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) row[R] = carry_s;
}
__global__ void csr_fill_kernel(const int *__restrict__ keys, long long total, int M, int R, int grp,
                                const int *__restrict__ offs, int *__restrict__ cursor, int *__restrict__ tmp)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const long long p = t / M;
    const int slot = (int)(t % M);
    const int key = keys[t];
    if (key < 0 || key >= R || csr_is_pad(keys, t, slot, key, grp)) return;
    const int pos = atomicAdd(cursor + p * (R + 1) + key, 1);
    tmp[p * M + offs[p * (R + 1) + key] + pos] = slot;
}
// order every bucket by slot id: rank = number of bucket members with a smaller slot
__global__ void csr_rank_kernel(const int *__restrict__ keys, long long total, int M, int R, int grp,
                                const int *__restrict__ offs, const int *__restrict__ tmp, int *__restrict__ perm)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const long long p = t / M;
    const int slot = (int)(t % M);
    const int key = keys[t];
    if (key < 0 || key >= R || csr_is_pad(keys, t, slot, key, grp)) return;
    const int lo = offs[p * (R + 1) + key], hi = offs[p * (R + 1) + key + 1];
    const int *b = tmp + p * M;
    int rank = 0;
    for (int e = lo; e < hi; ++e) rank += (b[e] < slot);
    perm[p * M + lo + rank] = slot;
}

// The same four steps for ONE problem per CTA with the bucket counters in shared memory (R <= 8192): one launch
// instead of two memsets + four kernels, shared-memory instead of L2 atomics.  Same deterministic output.
__global__ void __launch_bounds__(1024) csr_fused_kernel(const int *__restrict__ keys, int M, int R, int grp,
                                                         int *__restrict__ offs, int *__restrict__ perm, int *__restrict__ tmp)
{
    extern __shared__ int csr_sm[];
    __shared__ int wsum[32];
    __shared__ int carry_s;
    int *cnt = csr_sm, *cur = csr_sm + R + 1;
    const long long p = blockIdx.x;
    const int *kp = keys + p * M;
    int *tp = tmp + p * M, *pp = perm + p * M;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i <= R; i += 1024) { cnt[i] = 0; if (i < R) cur[i] = 0; }
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int e = threadIdx.x; e < M; e += 1024) {
        const int key = kp[e];
        if (key >= 0 && key < R && !csr_is_pad(kp, e, e, key, grp)) atomicAdd(cnt + key, 1);
    }
    __syncthreads();
    for (int base = 0; base < R; base += 1024) {               // exclusive scan, as csr_scan_kernel
        const int i = base + threadIdx.x;
        const int v = i < R ? cnt[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int sv = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, sv, o); if (lane >= o) sv += y; }
            wsum[lane] = sv;
        }
        __syncthreads();
        const int incl = x + (warp ? wsum[warp - 1] : 0) + carry_s;
        if (i < R) cnt[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) cnt[R] = carry_s;
    __syncthreads();
    int *op = offs + p * (R + 1);
    for (int i = threadIdx.x; i <= R; i += 1024) op[i] = cnt[i];
    // Fill in chunks of 1024 consecutive entries with a barrier between chunks: a bucket then holds its entries in
    // ascending CHUNK order, only the members of one chunk are in arrival order.  (Without it every entry had to be
    // ranked against its whole bucket: quadratic in the bucket size, 0.8 ms per step at N = 65536 where a coarse point
    // of FP1 collects ~190 entries.)
    for (int base = 0; base < M; base += 1024) {
        const int e = base + threadIdx.x;
        if (e < M) {
            const int key = kp[e];
            if (key >= 0 && key < R && !csr_is_pad(kp, e, e, key, grp)) {
                const int pos = atomicAdd(cur + key, 1);
                tp[cnt[key] + pos] = e;
            }
        }
        __syncthreads();
    }
    // order every bucket by entry id: find the run of this entry's chunk inside the bucket (binary search over the
    // chunk-sorted list), rank within the run
    for (int e = threadIdx.x; e < M; e += 1024) {
        const int key = kp[e];
        if (key < 0 || key >= R || csr_is_pad(kp, e, e, key, grp)) continue;
        const int lo = cnt[key], hi = cnt[key + 1];
        const int c = e >> 10;
        int a = lo, b = hi;                                   // first position whose chunk id is >= c
        while (a < b) {
            const int mid = (a + b) >> 1;
            if ((tp[mid] >> 10) < c) a = mid + 1; else b = mid;
        }
        int rank = 0;
        for (int q = a; q < hi; ++q) {
            const int o = tp[q];
            if ((o >> 10) != c) break;
            rank += (o < e);
        }
        pp[a + rank] = e;
    }
}

// ---- ordered segmented sum (backward of group / interp) ---------------------------------------
// dst[p*R + r][c] (+)= sum over bucket entries e (ascending slot) of scale_e * src[p*rows_per_p + slot_e/div][c]
// LPR lanes per destination row (narrow rows share a warp); the entry loop issues four independent
// loads at a time and adds them in bucket order, so the result is bit-reproducible.
template <int LPR>
__global__ void __launch_bounds__(256)
segsum_kernel(TView src, long long src_rows_per_p, int div, const float *__restrict__ wgt,
              const int *__restrict__ offs, const int *__restrict__ perm, int M, int R, long long P,
              int nch, int tail_cols, TView dst, int accumulate, TView rmask, const float *__restrict__ src_rm, int rm_stride)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");          // launched with programmatic stream serialization
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long wid = gid / LPR;                 // destination row
    const int lane = (int)(gid % LPR);
    if (wid >= P * R) return;
    const long long p = wid / R;
    const int r = (int)(wid % R);
    const int lo = offs[p * (R + 1) + r], hi = offs[p * (R + 1) + r + 1];
    const int *pm = perm + p * M;
    const float *ww = wgt ? wgt + p * M : nullptr;
    const long long sbase = p * src_rows_per_p;
    for (int c = lane; c < nch; c += LPR) {
        float4 acc = accumulate ? tv_ld(dst, wid, c) : make_float4(0.f, 0.f, 0.f, 0.f);
        const bool tail = (c == nch - 1 && tail_cols);
        for (int e = lo; e < hi; e += 4) {
            int slot[4]; float4 v[4]; float sc[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) slot[u] = e + u < hi ? pm[e + u] : -1;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                // src_rm: row-major copy of the source rows -- the lanes of one destination row then read one
                // contiguous piece of a source row (whole sectors) instead of 16-byte pieces 2 KB apart
                v[u] = slot[u] < 0 ? make_float4(0.f, 0.f, 0.f, 0.f)
                     : src_rm  ? *reinterpret_cast<const float4 *>(src_rm + (sbase + slot[u] / div) * rm_stride + 4 * c)
                               : tv_ld(src, sbase + slot[u] / div, c);
                sc[u] = (ww && slot[u] >= 0) ? ww[slot[u]] : 1.f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (slot[u] < 0) continue;
                float4 q = v[u];
                if (tail) {                      // keep only the first tail_cols of the last chunk
                    if (tail_cols < 2) q.y = 0.f;
                    if (tail_cols < 3) q.z = 0.f;
                    q.w = 0.f;
                }
                if (ww) {
                    acc.x = fmaf(q.x, sc[u], acc.x); acc.y = fmaf(q.y, sc[u], acc.y);
                    acc.z = fmaf(q.z, sc[u], acc.z); acc.w = fmaf(q.w, sc[u], acc.w);
                } else {
                    acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
                }
            }
        }
        if (rmask.base) {                          // gradient w.r.t. the pre-activation of a ReLU layer
            float4 y = tv_ld(rmask, wid, c);
            acc.x = y.x > 0.f ? acc.x : 0.f; acc.y = y.y > 0.f ? acc.y : 0.f;
            acc.z = y.z > 0.f ? acc.z : 0.f; acc.w = y.w > 0.f ? acc.w : 0.f;
        }
        tv_st(dst, wid, c, acc);
    }
}

// The same kernel specialised for the two callers that matter (ncu, warm caches: the generic kernel above is
// instruction-issue bound -- 66 % issue utilisation at 38 % occupancy, 87 warp instructions per bucket entry of which 4 are
// the FFMAs: a run-time integer division per entry, 64-bit address products, per-entry tail / weight / mirror branches):
//   INTERP: backward of the 3-NN interpolation (slot / 3, weighted, fmaf);  !INTERP: backward of the grouping gather
//   (slot, unweighted, add);  RM: sources are the row-major mirror.  Offsets inside a
// problem are 32-bit.  Same order of additions, same bits.
template <int LPR, bool INTERP, bool RM>
__global__ void __launch_bounds__(256)
segsum_fast_kernel(TView src, unsigned src_rows_per_p, const float *__restrict__ wgt, const int *__restrict__ offs,
                   const int *__restrict__ perm, int M, int R, long long P, int nch, TView dst, int accumulate, TView rmask,
                   const float *__restrict__ src_rm, unsigned rm_stride, int tail_cols)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");          // launched with programmatic stream serialization
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long wid = gid / LPR;                 // destination row
    const int lane = (int)(gid % LPR);
    if (wid >= P * R) return;
    const long long p = wid / R;
    const int r = (int)(wid - p * R);
    const int lo = offs[p * (R + 1) + r], hi = offs[p * (R + 1) + r + 1];
    const int *pm = perm + p * M;
    const float *ww = INTERP ? wgt + p * M : nullptr;
    // base of this problem's source rows: row-major mirror, or T-layout (whole problems start on 128-row tile boundaries
    // whenever rows_per_p % 128 == 0; otherwise the row offset is folded into the per-entry row)
    const float *rmb = RM ? src_rm + (size_t)p * src_rows_per_p * rm_stride : nullptr;
    const unsigned row0 = RM ? 0u : (unsigned)((p * src_rows_per_p) & 127);
    const float *tlb = RM ? nullptr : src.base + ((size_t)((p * src_rows_per_p) >> 7) * src.wchunks + src.c0) * 512;
    const unsigned wch = (unsigned)src.wchunks;
    for (int c = lane; c < nch; c += LPR) {
        const float4 acc0 = accumulate ? tv_ld(dst, wid, c) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 acc = acc0;
        constexpr int U = 4;          // entries in flight (8: measured slower; 8 CTAs per SM at 32 registers: within noise)
        for (int e = lo; e < hi; e += U) {
            unsigned srow[U]; float4 v[U]; float sc[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int sl = e + u < hi ? pm[e + u] : -1;
                if (INTERP) sc[u] = sl >= 0 ? ww[sl] : 0.f;
                srow[u] = sl < 0 ? 0xffffffffu : (INTERP ? (unsigned)sl / 3u : (unsigned)sl);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (srow[u] == 0xffffffffu) { v[u] = make_float4(0.f, 0.f, 0.f, 0.f); continue; }
                if (RM) v[u] = *reinterpret_cast<const float4 *>(rmb + srow[u] * rm_stride + 4u * (unsigned)c);
                else {
                    const unsigned rr = srow[u] + row0;
                    v[u] = *reinterpret_cast<const float4 *>(tlb + ((size_t)((rr >> 7) * wch + (unsigned)c) * 512u + (rr & 127u) * 4u));
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (srow[u] == 0xffffffffu) continue;
                if (INTERP) {
                    acc.x = fmaf(v[u].x, sc[u], acc.x); acc.y = fmaf(v[u].y, sc[u], acc.y);
                    acc.z = fmaf(v[u].z, sc[u], acc.z); acc.w = fmaf(v[u].w, sc[u], acc.w);
                } else {
                    acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
                }
            }
        }
        if (tail_cols && c == nch - 1) {           // columns past the tensor's width in the last chunk contribute nothing:
            if (tail_cols < 2) acc.y = acc0.y;     // what the generic kernel gets by zeroing them in every entry
            if (tail_cols < 3) acc.z = acc0.z;
            acc.w = acc0.w;
        }
        if (rmask.base) {                          // gradient w.r.t. the pre-activation of a ReLU layer
            float4 y = tv_ld(rmask, wid, c);
            acc.x = y.x > 0.f ? acc.x : 0.f; acc.y = y.y > 0.f ? acc.y : 0.f;
            acc.z = y.z > 0.f ? acc.z : 0.f; acc.w = y.w > 0.f ? acc.w : 0.f;
        }
        tv_st(dst, wid, c, acc);
    }
}

template <int LPR>
cudaError_t launch_segsum_fast(bool interp, bool rm, unsigned grid, cudaStream_t st, TView src, long long src_rows_per_p, const float *wgt,
                               const int *offs, const int *perm, int M, int R, long long P, int nch, TView dst, int accumulate, TView rmk,
                               const float *src_rm, int rm_stride, int tail)
{
    const unsigned rpp = (unsigned)src_rows_per_p, rs = (unsigned)rm_stride;
    if (interp && rm) return psg_launch_pdl(segsum_fast_kernel<LPR, true, true>, dim3(grid), dim3(256), 0, st, 1, src, rpp, wgt, offs, perm, M, R, P, nch, dst, accumulate, rmk, src_rm, rs, tail);
    if (interp) return psg_launch_pdl(segsum_fast_kernel<LPR, true, false>, dim3(grid), dim3(256), 0, st, 1, src, rpp, wgt, offs, perm, M, R, P, nch, dst, accumulate, rmk, src_rm, rs, tail);
    if (rm) return psg_launch_pdl(segsum_fast_kernel<LPR, false, true>, dim3(grid), dim3(256), 0, st, 1, src, rpp, wgt, offs, perm, M, R, P, nch, dst, accumulate, rmk, src_rm, rs, tail);
    return psg_launch_pdl(segsum_fast_kernel<LPR, false, false>, dim3(grid), dim3(256), 0, st, 1, src, rpp, wgt, offs, perm, M, R, P, nch, dst, accumulate, rmk, src_rm, rs, tail);
}

// dst[row][c] (+)= src[row][c] over a column slice
__global__ void copy_cols_kernel(TView src, TView dst, long long rows, int nch, int accumulate)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = t % rows;
    const int c = (int)(t / rows);
    if (c >= nch) return;
    float4 v = tv_ld(src, row, c);
    if (accumulate) { float4 d = tv_ld(dst, row, c); v.x += d.x; v.y += d.y; v.z += d.z; v.w += d.w; }
    tv_st(dst, row, c, v);
}

// ---- public row-major index_points -------------------------------------------------------------
__global__ void index_points_kernel(const float *__restrict__ pts, const long long *__restrict__ idx,
                                    int N, int C, long long M, long long total, float *__restrict__ out)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total * C) return;
    const long long e = t / C;
    const int ch = (int)(t % C);
    const long long b = e / M;
    const long long src = idx[e];
    out[t] = pts[(b * N + src) * C + ch];
}

// C % 4 == 0: one 128-bit load + store per thread, a gathered row is read and written as whole 16-byte pieces by
// consecutive threads (full sectors both ways); the index is read once per 16 bytes, not once per float
__global__ void index_points_v4_kernel(const float4 *__restrict__ pts, const long long *__restrict__ idx, int N, int C4, long long M,
                                       long long total, float4 *__restrict__ out)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total * C4) return;
    const long long e = t / C4;
    const int ch = (int)(t - e * C4);
    const long long b = e / M;
    const long long src = __ldg(idx + e);
    out[t] = __ldg(pts + (b * N + src) * C4 + ch);
}

inline unsigned nblocks(long long threads, int bs) { return (unsigned)((threads + bs - 1) / bs); }

}  // namespace

int psg_pack_cf(const float *x, long long sb, long long sc, long long sn, int B, int C, int N, TView out,
                int cpad, float *xyz, cudaStream_t st)
{
    pack_cf_kernel<<<nblocks((long long)B * N, 256), 256, 0, st>>>(x, sb, sc, sn, B, C, N, out, cpad, xyz);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_unpack_cf(TView in, int B, int C, int N, float *y, int accumulate, cudaStream_t st)
{
    unpack_cf_kernel<<<nblocks((long long)B * N, 256), 256, 0, st>>>(in, B, C, N, y, accumulate);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_pack_rm(const float *x, long long rows, int C, TView out, int cpad, cudaStream_t st)
{
    pack_rm_kernel<<<nblocks(rows * (cpad / 4), 256), 256, 0, st>>>(x, rows, C, out, cpad);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_unpack_rm(TView in, long long rows, int C, float *y, cudaStream_t st)
{
    unpack_rm_kernel<<<nblocks(rows * ((C + 3) / 4), 256), 256, 0, st>>>(in, rows, C, y);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_group(TView feats, int D, const float *xyz, long long cloud_stride, int nclouds, int Nsrc,
              const float *new_xyz, const int *idx, int P, int S, int K, TView out, int cpad, cudaStream_t st)
{
    const long long rows = (long long)P * S * K;
    group_kernel<<<nblocks(rows * (cpad / 4), 256), 256, 0, st>>>(feats, D, xyz, cloud_stride, nclouds, Nsrc,
                                                                   new_xyz, idx, P, S, K, out, cpad);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_maxpool(TView in, long long groups, int K, int C, TView out, unsigned char *arg, cudaStream_t st)
{
    if (K == 32) maxpool_kernel<32><<<nblocks(groups * 32 * (C / 4), 256), 256, 0, st>>>(in, groups, C, out, arg);
    else if (K == 16) maxpool_kernel<16><<<nblocks((groups + 1) / 2 * 32 * (C / 4), 256), 256, 0, st>>>(in, groups, C, out, arg);
    else return PSG_EUNSUPPORTED;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_maxpool_bwd(TView dout, TView outv, const unsigned char *arg, long long groups, int K, int C, TView dy,
                    cudaStream_t st)
{
    const long long th = groups * K * (C / 4);
    if (K == 32) maxpool_bwd_kernel<32><<<nblocks(th, 256), 256, 0, st>>>(dout, outv, arg, groups, C, dy);
    else if (K == 16) maxpool_bwd_kernel<16><<<nblocks(th, 256), 256, 0, st>>>(dout, outv, arg, groups, C, dy);
    else return PSG_EUNSUPPORTED;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_interp(TView feats, int S, const int *idx, const float *w, long long P, int N, int nch, TView out,
               cudaStream_t st)
{
    const long long rows = P * N;
    if (psg_launch_pdl(interp_kernel, dim3(nblocks(rows * nch, 256)), dim3(256), 0, st, 1, feats, S, idx, w, rows, N, nch, out) != cudaSuccess)
        return PSG_ECUDA;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
// offs [P][R+1], perm [P][M]; scratch: cursor [P][R+1] ints + tmp [P][M] ints
size_t psg_csr_scratch_bytes(long long P, int M, int R) { return (size_t)P * ((size_t)(R + 1) + M) * sizeof(int); }
int psg_csr_build(const int *keys, long long P, int M, int R, int grp, int *offs, int *perm, void *scratch,
                  cudaStream_t st)
{
    int *cursor = (int *)scratch;
    int *tmp = cursor + P * (R + 1);
    const long long total = P * M;
    if (R <= 8192) {
        const size_t smem = (size_t)(2 * R + 1) * sizeof(int);
        static PsgDeviceOnce attr_once;
        if (attr_once.need()) {
            if (cudaFuncSetAttribute(csr_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (2 * 8192 + 1) * 4) != cudaSuccess)
                return PSG_ECUDA;
            attr_once.mark();
        }
        csr_fused_kernel<<<(unsigned)P, 1024, smem, st>>>(keys, M, R, grp, offs, perm, tmp);
        PSG_LAUNCH_CHECK();
        return PSG_OK;
    }
    if (cudaMemsetAsync(offs, 0, (size_t)P * (R + 1) * sizeof(int), st) != cudaSuccess) return PSG_ECUDA;
    if (cudaMemsetAsync(cursor, 0, (size_t)P * (R + 1) * sizeof(int), st) != cudaSuccess) return PSG_ECUDA;
    csr_count_kernel<<<nblocks(total, 256), 256, 0, st>>>(keys, total, M, R, grp, offs);
    csr_scan_kernel<<<(unsigned)P, 1024, 0, st>>>(offs, R);
    csr_fill_kernel<<<nblocks(total, 256), 256, 0, st>>>(keys, total, M, R, grp, offs, cursor, tmp);
    csr_rank_kernel<<<nblocks(total, 256), 256, 0, st>>>(keys, total, M, R, grp, offs, tmp, perm);
    PSG_LAUNCH_CHECK();
    g_psg_launch_count += 3;
    return PSG_OK;
}
int psg_segsum(TView src, long long src_rows_per_p, int div, const float *wgt, const int *offs, const int *perm,
               int M, int R, long long P, int ncols, TView dst, int accumulate, const TView *relu_mask, const float *src_rm,
               int rm_stride, cudaStream_t st)
{
    TView rm = relu_mask ? *relu_mask : TView{nullptr, 0, 0};
    const int nch = (ncols + 3) / 4;
    cudaError_t err = cudaSuccess;
    if (((div == 3 && wgt) || (div == 1 && !wgt)) && src_rows_per_p < (1ll << 24) && (long long)M < (1ll << 30)) {
        // the two real callers (interpolation backward, gather backward): specialised kernel, same sums
        const bool interp = div == 3, rmm = src_rm != nullptr;
        const int lpr = nch <= 4 ? 4 : nch <= 8 ? 8 : nch <= 16 ? 16 : nch <= 32 ? 32 : nch <= 64 ? 64 : 128;
        const unsigned grid = nblocks(P * R * lpr, 256);
#define PSG_SF(L) launch_segsum_fast<L>(interp, rmm, grid, st, src, src_rows_per_p, wgt, offs, perm, M, R, P, nch, dst, accumulate, rm, src_rm, rm_stride, ncols & 3)
        err = lpr == 4 ? PSG_SF(4) : lpr == 8 ? PSG_SF(8) : lpr == 16 ? PSG_SF(16) : lpr == 32 ? PSG_SF(32) : lpr == 64 ? PSG_SF(64) : PSG_SF(128);
#undef PSG_SF
    } else if (nch <= 4)
        err = psg_launch_pdl(segsum_kernel<4>, dim3(nblocks(P * R * 4, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    else if (nch <= 8)
        err = psg_launch_pdl(segsum_kernel<8>, dim3(nblocks(P * R * 8, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    else if (nch <= 16)
        err = psg_launch_pdl(segsum_kernel<16>, dim3(nblocks(P * R * 16, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    else if (nch <= 32)
        err = psg_launch_pdl(segsum_kernel<32>, dim3(nblocks(P * R * 32, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    else if (nch <= 64)      // wide rows of the small levels: more lanes per row, the bucket walk is the latency chain
        err = psg_launch_pdl(segsum_kernel<64>, dim3(nblocks(P * R * 64, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    else
        err = psg_launch_pdl(segsum_kernel<128>, dim3(nblocks(P * R * 128, 256)), dim3(256), 0, st, 1, src, src_rows_per_p, div, wgt,
                             offs, perm, M, R, P, nch, ncols & 3, dst, accumulate, rm, src_rm, rm_stride);
    if (err != cudaSuccess) return PSG_ECUDA;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_copy_cols(TView src, TView dst, long long rows, int ncols, int accumulate, cudaStream_t st)
{
    const int nch = ncols / 4;
    copy_cols_kernel<<<nblocks(rows * nch, 256), 256, 0, st>>>(src, dst, rows, nch, accumulate);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
int psg_index_points_rm(const float *pts, const long long *idx, int B, int N, int C, long long M, float *out,
                        cudaStream_t st)
{
    const long long total = (long long)B * M;
    if (C % 4 == 0 && ((uintptr_t)pts & 15) == 0 && ((uintptr_t)out & 15) == 0) {
        index_points_v4_kernel<<<nblocks(total * (C / 4), 256), 256, 0, st>>>(reinterpret_cast<const float4 *>(pts), idx, N, C / 4, M,
                                                                             total, reinterpret_cast<float4 *>(out));
        PSG_LAUNCH_CHECK();
        return PSG_OK;
    }
    index_points_kernel<<<nblocks(total * C, 256), 256, 0, st>>>(pts, idx, N, C, M, total, out);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
