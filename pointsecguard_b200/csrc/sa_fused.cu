// sa_fused.cu -- set-abstraction level as ONE kernel per direction (tcgen05 TF32 mode).
//
// Reference: PointNet/models/pointnet_util.py:126-137 / :245-255 (gather neighbours, centre xyz,
// concat), :200-205 / :256-262 (three 1x1 conv + BN + ReLU layers, max over the K neighbours) and
// the autograd of the same.
//
// Forward, per 128-row tile (= 128/K neighbourhoods), persistent CTAs:
//   workers (4 warps, thread = tile row = TMEM lane) gather the grouped rows straight into shared
//   memory in the UMMA K-major no-swizzle operand layout; one MMA thread issues
//   tcgen05.mma.kind::tf32 against the folded weights, which stay resident in shared memory for the
//   CTA's lifetime; the workers read the accumulator back with tcgen05.ld, apply bias + ReLU and
//   write the next layer's A operand into shared memory; the last epilogue takes the max over each
//   neighbourhood with warp REDUX (a warp holds exactly 32/K neighbourhoods) and stores only the
//   pooled row and its arg-max.  The grouped tensor and the three activation tensors of the
//   unfused path (1.2 KB per row in SA1) never exist in HBM.
//
// Backward needs no activation VALUES (dgrad only, no wgrad): the forward keeps one ReLU bit per
// activation (8 B per row in SA1).  Per tile: scatter dOut to the arg-max rows -> dY2 in shared
// memory -> three dgrad GEMMs with the bit masks applied in the epilogues -> dG rows to HBM, which
// the deterministic segmented sum (gather.cu) then reduces by source point.
#include <cstdio>
#include "psg_common.cuh"
#include "psg_internal.h"
#include "psg_tc.cuh"
#include "psg_epi.cuh"

namespace {

constexpr int kWorkers = 128;

__device__ __forceinline__ float4 *plane_ptr(unsigned char *buf, int chunk, int row)
{
    return reinterpret_cast<float4 *>(buf) + (size_t)chunk * 128 + row;
}

// packed global weights [planes][nw][4] -> shared [planes][n][4]
__device__ __forceinline__ void load_weights(unsigned char *dst, const float *src, int planes, int n, int nw)
{
    float4 *d = reinterpret_cast<float4 *>(dst);
    const float4 *s = reinterpret_cast<const float4 *>(src);
    for (int e = threadIdx.x; e < planes * n; e += blockDim.x) {
        const int j = e / n, r = e - j * n;
        d[e] = __ldg(s + (size_t)j * nw + r);
    }
}

// D[128 x n] (+)= A[128 x 4*planes] * B[n x 4*planes]^T, both operands in shared memory
__device__ __forceinline__ void issue_layer(uint32_t tmem, uint32_t sA, uint32_t sB, int planes, int n, uint32_t acc = 0)
{
    const uint32_t idesc = tc::idesc_tf32(128, n);
    for (int j = 0; j < planes; j += 2) {
        const uint64_t ad = tc::smem_desc(sA + j * 2048, 2048, 128);
        const uint64_t bd = tc::smem_desc(sB + j * n * 16, (uint32_t)(n * 16), 128);
        tc::mma_tf32(tmem, ad, bd, idesc, acc);
        acc = 1;
    }
}

// 3xTF32 (X3 kernels): kind::tf32 reads the top 19 bits of an operand, so a value as it lies in shared memory is its own
// "hi" part; lo4 is what the hardware drops (exact in fp32), written to a second operand buffer.  Three MMAs per K step
// -- A_lo W_hi + A_hi W_lo + A_hi W_hi -- give fp32-grade products (gemm_tc.cu has the per-layer twin).
__device__ __forceinline__ float4 lo4(float4 a)
{
    float4 l;
    l.x = a.x - __uint_as_float(__float_as_uint(a.x) & 0xFFFFE000u);
    l.y = a.y - __uint_as_float(__float_as_uint(a.y) & 0xFFFFE000u);
    l.z = a.z - __uint_as_float(__float_as_uint(a.z) & 0xFFFFE000u);
    l.w = a.w - __uint_as_float(__float_as_uint(a.w) & 0xFFFFE000u);
    return l;
}
__device__ __forceinline__ void issue_layer_x3(uint32_t tmem, uint32_t sA, uint32_t sAl, uint32_t sBh, uint32_t sBl, int planes, int n,
                                               uint32_t acc = 0)
{
    const uint32_t idesc = tc::idesc_tf32(128, n);
    for (int j = 0; j < planes; j += 2) {
        const uint64_t ad = tc::smem_desc(sA + j * 2048, 2048, 128), al = tc::smem_desc(sAl + j * 2048, 2048, 128);
        const uint64_t bh = tc::smem_desc(sBh + j * n * 16, (uint32_t)(n * 16), 128), bl = tc::smem_desc(sBl + j * n * 16, (uint32_t)(n * 16), 128);
        tc::mma_tf32(tmem, al, bh, idesc, acc);      // small terms first
        tc::mma_tf32(tmem, ad, bl, idesc, 1u);
        tc::mma_tf32(tmem, ad, bh, idesc, 1u);
        acc = 1;
    }
}

__device__ __forceinline__ long long gtimer()
{
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

struct SaFwdArgs {
    TView feats; int D; const float *xyz; long long cloud_stride; int nclouds; int Nsrc;
    const float *new_xyz; const int *idx; long long rows; int S;
    int gpad, n0, n1, n2;
    const float *w0, *w1, *w2; int nw0, nw1, nw2;
    const float *b0, *b1, *b2;
    unsigned *m0, *m1;
    TView out; unsigned char *arg;
    int ntiles;
    long long *trace;
    const int *crow_src, *crow_g, *ntiles_dev;      // compacted rows (compact.cu); CP kernels only
    const float *w0l, *w1l, *w2l;                   // X3 kernels: the TF32 residuals of w0..w2 (same packing)
};

// accumulator -> bias + ReLU -> next A operand in shared memory (+ one ReLU bit per element)
template <bool X3 = false>
__device__ __forceinline__ void epilogue_relu_to_smem(uint32_t tmem_lane, int n, const float *bias,
                                                      unsigned char *dst, unsigned *mask_tile, int row, unsigned char *dst_lo = nullptr)
{
    int c = 0;
    for (; c + 32 <= n; c += 32) {
        float v[32];
        tc::tmem_ld32(tmem_lane + (uint32_t)c, v);
        const unsigned w = psg_relu_bias_bits<32>(v, bias + c);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 y = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            *plane_ptr(dst, (c >> 2) + q, row) = y;
            if (X3) *plane_ptr(dst_lo, (c >> 2) + q, row) = lo4(y);
        }
        mask_tile[(size_t)(c >> 5) * 128 + row] = w;
    }
    if (c < n) {
        float v[16];
        tc::tmem_ld16(tmem_lane + (uint32_t)c, v);
        const unsigned w = psg_relu_bias_bits<16>(v, bias + c);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 y = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            *plane_ptr(dst, (c >> 2) + q, row) = y;
            if (X3) *plane_ptr(dst_lo, (c >> 2) + q, row) = lo4(y);
        }
        mask_tile[(size_t)(c >> 5) * 128 + row] = w;
    }
}

// CP: the rows are the compacted real hits (compact.cu) -- source point and centroid come from crow_src / crow_g, the tile
// count from device memory, and the pool scans variable-length segments of the warp's four octets.
template <int K, int NG, bool CP, bool X3 = false>
__global__ void __launch_bounds__(NG * 160, NG == 1 ? 4 : (NG == 2 ? 2 : 1)) sa_fwd_kernel(SaFwdArgs a)
{
    static_assert(!X3 || CP, "the 3xTF32 kernels run on compacted rows only");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar_in[NG], bar_acc[NG];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float sbias[3][128];      // folded biases: epilogues read them with broadcast LDS

    const uint32_t s0 = tc::smem_u32(smem_raw);
    const uint32_t sbase = (s0 + 1023u) & ~1023u;
    unsigned char *base = smem_raw + (sbase - s0);
    const int szW0 = a.gpad * a.n0 * 4, szW1 = a.n0 * a.n1 * 4, szW2 = (a.n1 * a.n2 * 4 + 1023) & ~1023;
    // per tile ONE operand buffer: a layer's MMA has completed before its epilogue runs, so the
    // epilogue overwrites the layer's own input in place (gather -> Y0 -> Y1)
    // (compacted rows: the segmented pool borrows 4 KB of the buffer per warp, so narrow branches get at least 16 KB)
    const int szG = CP ? max(max(a.gpad, max(a.n0, a.n1)) * 512, 16384) : max(a.gpad, max(a.n0, a.n1)) * 512;
    // X3: [W hi x3][W lo x3][per tile: A | A_lo]
    const int szWall = szW0 + szW1 + szW2;
    unsigned char *pW0 = base, *pW1 = pW0 + szW0, *pW2 = pW1 + szW1, *pG = pW2 + szW2 + (X3 ? szWall : 0);
    const uint32_t sW0 = sbase, sW1 = sW0 + szW0, sW2 = sW1 + szW1, sG = sW2 + szW2 + (X3 ? szWall : 0);
    const int tileG = X3 ? 2 * szG : szG;            // operand bytes per tile in flight

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    long long *gtr = (a.trace && threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
                         ? a.trace + 3 * 512 + (blockIdx.x ? 8 : 0) : nullptr;
    if (gtr) gtr[0] = gtimer();
    const int nmax = max(a.n0, max(a.n1, a.n2));
    const uint32_t gcols = tc::next_pow2_cols(nmax);       // TMEM columns per group
    const uint32_t ncols = tc::next_pow2_cols((int)(gcols * NG));   // tcgen05.alloc takes powers of two

    load_weights(pW0, a.w0, a.gpad / 4, a.n0, a.nw0);
    load_weights(pW1, a.w1, a.n0 / 4, a.n1, a.nw1);
    load_weights(pW2, a.w2, a.n1 / 4, a.n2, a.nw2);
    if (X3) {
        load_weights(pW0 + szWall, a.w0l, a.gpad / 4, a.n0, a.nw0);
        load_weights(pW1 + szWall, a.w1l, a.n0 / 4, a.n1, a.nw1);
        load_weights(pW2 + szWall, a.w2l, a.n1 / 4, a.n2, a.nw2);
    }
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
        sbias[0][i] = i < a.n0 ? __ldg(a.b0 + i) : 0.f;
        sbias[1][i] = i < a.n1 ? __ldg(a.b1 + i) : 0.f;
        sbias[2][i] = i < a.n2 ? __ldg(a.b2 + i) : 0.f;
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            tc::mbar_init(tc::smem_u32(&bar_in[g]), kWorkers);
            tc::mbar_init(tc::smem_u32(&bar_acc[g]), 1);
        }
        tc::fence_mbar_init();
    }
    if (warp == NG * 4) tc::tmem_alloc(tc::smem_u32(&tmem_slot), ncols);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (gtr) gtr[1] = gtimer();
    tc::pdl_launch_dependents();      // the next kernel's prologue may overlap our tail ...
    tc::pdl_wait();                   // ... and ours overlapped our predecessor's: wait for its results now
    if (gtr) gtr[2] = gtimer();
    const uint32_t tmem = tmem_slot;
    const int tstride = gridDim.x * NG;
    const int ntiles = CP ? __ldg(a.ntiles_dev) : a.ntiles;

    if (warp >= NG * 4) {
        if (lane == 0) {
            // ---- MMA issuers: one warp per tile in flight, so that a group's next layer never queues behind
            // the other groups' issue work (a single polling thread cost ~1000 cycles per layer at NG = 4) ----
            const int g = warp - NG * 4;
            const uint32_t b_in = tc::smem_u32(&bar_in[g]), b_acc = tc::smem_u32(&bar_acc[g]);
            const uint32_t sA = sG + g * tileG, tm = tmem + g * gcols;
            uint32_t ph = 0;
            for (int tile = blockIdx.x * NG + g; tile < ntiles; tile += tstride) {
#pragma unroll 1
                for (int layer = 0; layer < 3; ++layer) {
                    tc::mbar_spin(b_in, ph); ph ^= 1u;
                    tc::fence_after_sync();
                    if (X3) {
                        if (layer == 0) issue_layer_x3(tm, sA, sA + szG, sW0, sW0 + szWall, a.gpad / 4, a.n0);
                        else if (layer == 1) issue_layer_x3(tm, sA, sA + szG, sW1, sW1 + szWall, a.n0 / 4, a.n1);
                        else issue_layer_x3(tm, sA, sA + szG, sW2, sW2 + szWall, a.n1 / 4, a.n2);
                    } else
                    if (layer == 0) issue_layer(tm, sA, sW0, a.gpad / 4, a.n0);
                    else if (layer == 1) issue_layer(tm, sA, sW1, a.n0 / 4, a.n1);
                    else issue_layer(tm, sA, sW2, a.n1 / 4, a.n2);
                    tc::mma_commit(b_acc);
                }
            }
        }
    } else {
        const int grp = warp >> 2, wq = warp & 3;
        const int r = threadIdx.x & 127;                 // tile row = TMEM lane
        unsigned char *pA = pG + (size_t)grp * tileG, *pY0 = pA, *pAl = pA + szG;
        const uint32_t b_in = tc::smem_u32(&bar_in[grp]), b_acc = tc::smem_u32(&bar_acc[grp]);
        const uint32_t tl = tmem + grp * gcols + ((uint32_t)(wq * 32) << 16);
        const int k = r % K;
        const unsigned gmask = (K == 32) ? 0xffffffffu : (0xffffu << (16 * ((lane / 16))));
        const int w0words = (a.n0 + 31) / 32, w1words = (a.n1 + 31) / 32;
        uint32_t ph = 0;
        long long *tr = (a.trace && blockIdx.x == 0 && r == 0 && grp < 2) ? a.trace + grp * 512 : nullptr;
        int tn = 0;
#define SA_STAMP() do { if (tr && tn < 510) tr[tn++] = clock64(); } while (0)
        SA_STAMP();
        int tile = blockIdx.x * NG + grp;
        int src_next = CP ? (tile < ntiles ? a.crow_src[(long long)tile * 128 + r] : -1)
                          : ((tile < ntiles && (long long)tile * 128 + r < a.rows) ? a.idx[(long long)tile * 128 + r] : 0);
        for (; tile < ntiles; tile += tstride) {
            const long long row = (long long)tile * 128 + r;
            const bool valid = CP ? src_next >= 0 : row < a.rows;
            const int cg = CP ? (valid ? a.crow_g[row] : -1) : 0;         // centroid of a compacted row
            // ---- gather: [ feats[src] (D) | xyz[src] - centre (3) | 0 ] -> A operand ----
            {
                const long long rr = valid ? row : 0;
                const long long ps = CP ? (valid ? cg : 0) : rr / K;
                const int p = (int)(ps / a.S);
                const int src = valid ? src_next : 0;
                const int cloud = p % a.nclouds;
                const long long srow = (long long)cloud * a.Nsrc + src;
                const int D = a.D;
                const int nfull = D >> 2;                 // chunks that are features only
#pragma unroll 8
                for (int c = 0; c < nfull; ++c) {
                    float4 v = valid ? tv_ld(a.feats, srow, c) : make_float4(0.f, 0.f, 0.f, 0.f);
                    *plane_ptr(pA, c, r) = v;
                    if (X3) *plane_ptr(pAl, c, r) = lo4(v);
                }
                const float *sp = a.xyz + (long long)cloud * a.cloud_stride + (long long)src * 3;
                const float *cp = a.new_xyz + ps * 3;
                const float dx = __fsub_rn(sp[0], cp[0]), dy = __fsub_rn(sp[1], cp[1]), dz = __fsub_rn(sp[2], cp[2]);
                for (int c = nfull; c < a.gpad / 4; ++c) {
                    float f[4] = {0.f, 0.f, 0.f, 0.f};
                    if (4 * c < D) { float4 q = tv_ld(a.feats, srow, c); f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w; }
                    float o[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int ch = 4 * c + j;
                        o[j] = ch < D ? f[j] : (ch == D ? dx : (ch == D + 1 ? dy : (ch == D + 2 ? dz : 0.f)));
                        if (!valid) o[j] = 0.f;
                    }
                    *plane_ptr(pA, c, r) = make_float4(o[0], o[1], o[2], o[3]);
                    if (X3) *plane_ptr(pAl, c, r) = lo4(make_float4(o[0], o[1], o[2], o[3]));
                }
                // prefetch the next tile's neighbour index: takes one L2 round trip off its gather
                const long long nrow = row + (long long)tstride * 128;
                if (CP) src_next = (tile + tstride < ntiles) ? a.crow_src[nrow] : -1;
                else src_next = (nrow < a.rows) ? a.idx[nrow] : 0;
            }
            tc::fence_async_smem();
            tc::mbar_arrive(b_in);
            SA_STAMP();
            // ---- layer 0 epilogue -> Y0 ----
            tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();
            SA_STAMP();
            epilogue_relu_to_smem<X3>(tl, a.n0, sbias[0], pY0, a.m0 + (size_t)tile * w0words * 128, r, pAl);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::mbar_arrive(b_in);
            SA_STAMP();
            // ---- layer 1 epilogue -> Y1 (reuses the gather buffer) ----
            tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();
            SA_STAMP();
            epilogue_relu_to_smem<X3>(tl, a.n1, sbias[1], pA, a.m1 + (size_t)tile * w1words * 128, r, pAl);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::mbar_arrive(b_in);
            SA_STAMP();
            // ---- layer 2 epilogue: bias + ReLU + max over the K rows of each neighbourhood ----
            tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();
            SA_STAMP();
            const long long g = row / K;
            if (CP) {
                // compacted rows: the warp's four octets form 1..4 neighbourhoods of 8..32 rows (compact.cu)
                float *scratch = reinterpret_cast<float *>(pA + (size_t)wq * 4096);
                int gq[4];
                unsigned sm, vm;
                psg_slice_segments(cg, gq, sm, vm);
                int c = 0;
                for (; c + 32 <= a.n2; c += 32) {
                    float v[32];
                    tc::tmem_ld32(tl + (uint32_t)c, v);
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + sbias[2][c + i], 0.f);
                    const int col = c + lane;
                    psg_pool_segmented<32>(v, scratch, lane, gq, sm, vm, [&](int gg, float best, int arg) {
                        a.out.base[tv_off(a.out, gg, col >> 2) + (col & 3)] = best;
                        a.arg[(long long)gg * a.n2 + col] = (unsigned char)arg;
                    });
                }
                if (c < a.n2) {
                    float v[16];
                    tc::tmem_ld16(tl + (uint32_t)c, v);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i] + sbias[2][c + i], 0.f);
                    const int col = c + lane;
                    psg_pool_segmented<16>(v, scratch, lane, gq, sm, vm, [&](int gg, float best, int arg) {
                        a.out.base[tv_off(a.out, gg, col >> 2) + (col & 3)] = best;
                        a.arg[(long long)gg * a.n2 + col] = (unsigned char)arg;
                    });
                }
            } else if (szG >= 16384) {
                // transposed pool: the tile's operand buffer is dead once MMA 2 has completed (every warp of
                // the tile waited on the same barrier), so warp wq borrows 4 KB of it as scratch
                float *scratch = reinterpret_cast<float *>(pA + (size_t)wq * 4096);
                const long long g0 = ((long long)tile * 128 + wq * 32) / K;          // first neighbourhood of this warp
                auto emit = [&](int col, const float *best, const int *arg) {
#pragma unroll
                    for (int gi = 0; gi < 32 / K; ++gi) {
                        const long long gg = g0 + gi;
                        if (gg * K < a.rows) {
                            a.out.base[tv_off(a.out, gg, col >> 2) + (col & 3)] = best[gi];
                            a.arg[gg * a.n2 + col] = (unsigned char)arg[gi];
                        }
                    }
                };
                int c = 0;
                for (; c + 32 <= a.n2; c += 32) {
                    float v[32];
                    tc::tmem_ld32(tl + (uint32_t)c, v);
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + sbias[2][c + i], 0.f);
                    float best[32 / K]; int arg[32 / K];
                    psg_pool_transposed<K, 32>(v, scratch, lane, best, arg);
                    emit(c + lane, best, arg);
                }
                if (c < a.n2) {
                    float v[16];
                    tc::tmem_ld16(tl + (uint32_t)c, v);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i] + sbias[2][c + i], 0.f);
                    float best[32 / K]; int arg[32 / K];
                    psg_pool_transposed<K, 16>(v, scratch, lane, best, arg);
                    if (lane < 16) emit(c + lane, best, arg);
                }
            } else
            for (int c16 = 0; c16 < a.n2; c16 += 16) {
                float v[16];
                tc::tmem_ld16(tl + (uint32_t)c16, v);
                unsigned am[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const unsigned b = __float_as_uint(fmaxf(v[i] + sbias[2][c16 + i], 0.f));
                    const unsigned mx = __reduce_max_sync(gmask, b);     // post-ReLU values order like their bits
                    am[i] = __reduce_min_sync(gmask, b == mx ? (unsigned)k : 64u);   // first arg-max
                    v[i] = __uint_as_float(mx);
                }
                if (k == 0 && valid) {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        tv_st(a.out, g, (c16 >> 2) + c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
                    uint4 pk;
                    pk.x = am[0] | (am[1] << 8) | (am[2] << 16) | (am[3] << 24);
                    pk.y = am[4] | (am[5] << 8) | (am[6] << 16) | (am[7] << 24);
                    pk.z = am[8] | (am[9] << 8) | (am[10] << 16) | (am[11] << 24);
                    pk.w = am[12] | (am[13] << 8) | (am[14] << 16) | (am[15] << 24);
                    *reinterpret_cast<uint4 *>(a.arg + g * a.n2 + c16) = pk;
                }
            }
            SA_STAMP();
            tc::fence_before_sync();
            // The transposed pool borrows WHOLE planes of the tile's operand buffer as per-warp scratch, and the next
            // tile's gather writes this warp's rows of EVERY plane: a warp that ran ahead would scribble over the scratch
            // of a sibling still pooling (seen as a rare run-to-run difference of a 50-step attack).  The four warps of
            // a tile meet here first (named barrier per tile in flight; they meet again at the next MMA hand-off anyway).
            if (CP || szG >= 16384) asm volatile("bar.sync %0, 128;" ::"r"(grp + 1) : "memory");
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (gtr) gtr[3] = gtimer();
    if (warp == NG * 4) tc::tmem_dealloc(tmem, ncols);
}

// ---------------------------------------------------------------------------------------------
struct SaBwdArgs {
    TView dout, outv; const unsigned char *arg;
    const unsigned *m0, *m1;
    const float *wb0, *wb1, *wb2; int nwb0, nwb1, nwb2;   // dgrad weights [cout/4][nwb][4], rows = cin
    TView dG; int gcols;
    float *dG_rm; int rm_only;    // row-major copy of the gradient rows ([rows][gpad]) for the segmented sum
    int slab;                 // columns of dY2 scattered per pass (n2 is contracted in n2 / slab passes)
    long long rows;
    int gpad, n0, n1, n2;
    int ntiles;
    long long *trace;
    const int *crow_g, *ntiles_dev;                 // compacted rows (compact.cu); CP kernels only
    const float *wb0l, *wb1l, *wb2l;                // X3 kernels: the TF32 residuals of the dgrad weights
};

// accumulator -> ReLU-bit mask -> next A operand in shared memory
template <bool X3 = false>
__device__ __forceinline__ void epilogue_mask_to_smem(uint32_t tmem_lane, int n, const unsigned *mask_tile,
                                                      unsigned char *dst, int row, unsigned char *dst_lo = nullptr)
{
    int c = 0;
    for (; c + 32 <= n; c += 32) {
        const unsigned w = mask_tile[(size_t)(c >> 5) * 128 + row];
        float v[32];
        tc::tmem_ld32(tmem_lane + (uint32_t)c, v);
        psg_apply_bits<32>(v, w);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 y = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            *plane_ptr(dst, (c >> 2) + q, row) = y;
            if (X3) *plane_ptr(dst_lo, (c >> 2) + q, row) = lo4(y);
        }
    }
    if (c < n) {
        const unsigned w = mask_tile[(size_t)(c >> 5) * 128 + row];
        float v[16];
        tc::tmem_ld16(tmem_lane + (uint32_t)c, v);
        psg_apply_bits<16>(v, w);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 y = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            *plane_ptr(dst, (c >> 2) + q, row) = y;
            if (X3) *plane_ptr(dst_lo, (c >> 2) + q, row) = lo4(y);
        }
    }
}

template <int K, int NG, bool CP, bool X3 = false>
__global__ void __launch_bounds__(NG * 160, NG == 1 ? 4 : (NG == 2 ? 2 : 1)) sa_bwd_kernel(SaBwdArgs a)
{
    static_assert(!X3 || CP, "the 3xTF32 kernels run on compacted rows only");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar_in[NG], bar_acc[NG];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float4 stg_d[NG * 4][32];      // per-warp staging of the arg-max scatter (psg_epi.cuh)
    __shared__ uchar4 stg_a[NG * 4][32];

    const uint32_t s0 = tc::smem_u32(smem_raw);
    const uint32_t sbase = (s0 + 1023u) & ~1023u;
    unsigned char *base = smem_raw + (sbase - s0);
    // dgrad weights of layer l: planes = cout_l / 4, rows = cin_l
    const int szW2 = a.n2 * a.n1 * 4, szW1 = a.n1 * a.n0 * 4, szW0 = (a.n0 * a.gpad * 4 + 1023) & ~1023;
    // per tile ONE operand buffer, overwritten in place: dY2 (one slab at a time) -> dY1 -> dY0
    const int szG = max(a.slab, max(a.n1, a.n0)) * 512;
    const int nslab = a.n2 / a.slab;
    // X3: [W hi x3][W lo x3][per tile: D | D_lo]
    const int szWall = szW2 + szW1 + szW0;
    unsigned char *pW2 = base, *pW1 = pW2 + szW2, *pW0 = pW1 + szW1, *pG = pW0 + szW0 + (X3 ? szWall : 0);
    const uint32_t sW2 = sbase, sW1 = sW2 + szW2, sW0 = sW1 + szW1, sG = sW0 + szW0 + (X3 ? szWall : 0);
    const int tileG = X3 ? 2 * szG : szG;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nmax = max(a.n0, max(a.n1, a.gpad));
    const uint32_t gcols = tc::next_pow2_cols(nmax);
    const uint32_t ncols = tc::next_pow2_cols((int)(gcols * NG));   // tcgen05.alloc takes powers of two

    load_weights(pW2, a.wb2, a.n2 / 4, a.n1, a.nwb2);
    load_weights(pW1, a.wb1, a.n1 / 4, a.n0, a.nwb1);
    load_weights(pW0, a.wb0, a.n0 / 4, a.gpad, a.nwb0);
    if (X3) {
        load_weights(pW2 + szWall, a.wb2l, a.n2 / 4, a.n1, a.nwb2);
        load_weights(pW1 + szWall, a.wb1l, a.n1 / 4, a.n0, a.nwb1);
        load_weights(pW0 + szWall, a.wb0l, a.n0 / 4, a.gpad, a.nwb0);
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            tc::mbar_init(tc::smem_u32(&bar_in[g]), kWorkers);
            tc::mbar_init(tc::smem_u32(&bar_acc[g]), 1);
        }
        tc::fence_mbar_init();
    }
    if (warp == NG * 4) tc::tmem_alloc(tc::smem_u32(&tmem_slot), ncols);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    tc::pdl_launch_dependents();      // the next kernel's prologue may overlap our tail ...
    tc::pdl_wait();                   // ... and ours overlapped our predecessor's: wait for its results now
    const uint32_t tmem = tmem_slot;
    const int tstride = gridDim.x * NG;
    const int ntiles = CP ? __ldg(a.ntiles_dev) : a.ntiles;

    if (warp >= NG * 4) {
        if (lane == 0) {
            // ---- MMA issuers: one warp per tile in flight (see sa_fwd_kernel) ----
            const int g = warp - NG * 4;
            const uint32_t b_in = tc::smem_u32(&bar_in[g]), b_acc = tc::smem_u32(&bar_acc[g]);
            const uint32_t sD = sG + g * tileG, tm = tmem + g * gcols;
            uint32_t ph = 0;
            for (int tile = blockIdx.x * NG + g; tile < ntiles; tile += tstride) {
#pragma unroll 1
                for (int L = 0; L < nslab + 2; ++L) {
                    tc::mbar_spin(b_in, ph); ph ^= 1u;
                    tc::fence_after_sync();
                    if (X3) {
                        const uint32_t w2off = (uint32_t)L * (a.slab / 4) * a.n1 * 16;
                        if (L < nslab) issue_layer_x3(tm, sD, sD + szG, sW2 + w2off, sW2 + szWall + w2off, a.slab / 4, a.n1, L > 0 ? 1u : 0u);
                        else if (L == nslab) issue_layer_x3(tm, sD, sD + szG, sW1, sW1 + szWall, a.n1 / 4, a.n0);
                        else issue_layer_x3(tm, sD, sD + szG, sW0, sW0 + szWall, a.n0 / 4, a.gpad);
                    } else
                    if (L < nslab)                                                        // dY1 (+)= dY2[:, slab L] W2[slab L]
                        issue_layer(tm, sD, sW2 + (uint32_t)L * (a.slab / 4) * a.n1 * 16, a.slab / 4, a.n1, L > 0 ? 1u : 0u);
                    else if (L == nslab) issue_layer(tm, sD, sW1, a.n1 / 4, a.n0);        // dY0 = dY1 W1
                    else issue_layer(tm, sD, sW0, a.n0 / 4, a.gpad);                     // dG  = dY0 W0
                    tc::mma_commit(b_acc);
                }
            }
        }
    } else {
        const int grp = warp >> 2, wq = warp & 3;
        const int r = threadIdx.x & 127;
        unsigned char *pD2 = pG + (size_t)grp * tileG, *pD1 = pD2, *pD0 = pD2, *pDl = pD2 + szG;
        const uint32_t b_in = tc::smem_u32(&bar_in[grp]), b_acc = tc::smem_u32(&bar_acc[grp]);
        const uint32_t tl = tmem + grp * gcols + ((uint32_t)(wq * 32) << 16);
        const int w0words = (a.n0 + 31) / 32, w1words = (a.n1 + 31) / 32;
        uint32_t ph = 0;
        long long *tr = (a.trace && blockIdx.x == 0 && r == 0 && grp < 2) ? a.trace + grp * 512 : nullptr;
        int tn = 0;
        SA_STAMP();
        for (int tile = blockIdx.x * NG + grp; tile < ntiles; tile += tstride) {
            const long long row = (long long)tile * 128 + r;
            const int cg = CP ? a.crow_g[row] : 0;
            const bool valid = CP ? cg >= 0 : row < a.rows;
            const long long g = CP ? (valid ? cg : 0) : (valid ? row : 0) / K;
            int rank = lane % K;
            if (CP) {
                // rank inside the neighbourhood: rows since the first octet that carries the same centroid
                int gq[4];
                unsigned sm, vm;
                psg_slice_segments(cg, gq, sm, vm);
                int f = lane >> 3;
#pragma unroll
                for (int u = 0; u < 3; ++u)
                    if (f > 0 && !((sm >> f) & 1u)) --f;
                rank = lane - 8 * f;
            }
            // ---- dY2[(g,k)][c] = (k == arg[g][c] && out[g][c] > 0) ? dOut[g][c] : 0, one slab of columns at a
            // time: the operand buffer stays small (more tiles in flight), the MMA accumulates over slabs ----
            for (int sl = 0; sl < nslab; ++sl) {
                if (CP)
                    psg_scatter_warp_rank<8>(a.dout, a.outv, a.arg, a.n2, g, valid, lane, rank, sl * (a.slab / 4), a.slab / 4,
                                             stg_d[warp], stg_a[warp], [&](int c, float4 q) {
                                                 *plane_ptr(pD2, c, r) = q;
                                                 if (X3) *plane_ptr(pDl, c, r) = lo4(q);
                                             });
                else
                psg_scatter_warp<K>(a.dout, a.outv, a.arg, a.n2, g, valid, lane, sl * (a.slab / 4), a.slab / 4,
                                    stg_d[warp], stg_a[warp], [&](int c, float4 q) { *plane_ptr(pD2, c, r) = q; });
                tc::fence_before_sync();
                tc::fence_async_smem();
                tc::mbar_arrive(b_in);
                SA_STAMP();
                tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();     // this slab's MMAs are done
                SA_STAMP();
            }
            epilogue_mask_to_smem<X3>(tl, a.n1, a.m1 + (size_t)tile * w1words * 128, pD1, r, pDl);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::mbar_arrive(b_in);
            SA_STAMP();
            tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();
            SA_STAMP();
            epilogue_mask_to_smem<X3>(tl, a.n0, a.m0 + (size_t)tile * w0words * 128, pD0, r, pDl);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::mbar_arrive(b_in);
            SA_STAMP();
            tc::mbar_wait(b_acc, ph); ph ^= 1u; tc::fence_after_sync();
            SA_STAMP();
            for (int c16 = 0; c16 < a.gcols; c16 += 16) {
                float v[16];
                tc::tmem_ld16(tl + (uint32_t)c16, v);
                if (valid) {
                    if (!a.rm_only) {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            tv_st(a.dG, row, (c16 >> 2) + c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
                    }
                    if (a.dG_rm) {
                        float4 *d = reinterpret_cast<float4 *>(a.dG_rm + row * a.gpad + c16);
#pragma unroll
                        for (int c = 0; c < 4; ++c) d[c] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                    }
                }
            }
            SA_STAMP();
            tc::fence_before_sync();
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == NG * 4) tc::tmem_dealloc(tmem, ncols);
}

int g_num_sms = 0;
constexpr size_t kSmemPerCtaMax = 224 * 1024;

inline size_t r1k(size_t x) { return (x + 1023) & ~(size_t)1023; }
inline int max3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }
inline size_t fwd_smem(int gpad, int n0, int n1, int n2, int ng, bool cp = false, bool x3 = false)
{
    size_t g = (size_t)max3(gpad, n0, n1) * 512;
    if (cp && g < 16384) g = 16384;              // the segmented pool's per-warp scratch lives in the operand buffer
    const size_t w = (size_t)gpad * n0 * 4 + (size_t)n0 * n1 * 4 + r1k((size_t)n1 * n2 * 4);
    return (x3 ? 2 : 1) * (w + (size_t)ng * g) + 1024;      // 3xTF32: hi and lo copies of the weights and of every operand buffer
}
// columns of dY2 scattered per pass: the largest 16-multiple divisor of n2 not wider than the hidden layers
// (the operand buffer has to hold those anyway)
inline int bwd_slab(int n0, int n1, int n2)
{
    const int cap = n0 > n1 ? n0 : n1;
    for (int sl = cap - cap % 16; sl >= 16; sl -= 16)
        if (n2 % sl == 0) return sl;
    return n2;
}
inline size_t bwd_smem_slab(int gpad, int n0, int n1, int n2, int ng, int slab, bool x3 = false)
{
    return (x3 ? 2 : 1) * ((size_t)n2 * n1 * 4 + (size_t)n1 * n0 * 4 + r1k((size_t)n0 * gpad * 4) +
                           (size_t)ng * (size_t)max3(slab, n1, n0) * 512) + 1024;
}
// The register file, not shared memory, limits a SM to about four tiles in flight, so when four whole-width
// operand buffers fit the scatter goes in ONE pass: every extra slab is one more MMA round trip (~1 us) per tile.
inline int bwd_slab_for(int gpad, int n0, int n1, int n2, bool x3 = false)
{
    if (bwd_smem_slab(gpad, n0, n1, n2, 4, n2, x3) <= kSmemPerCtaMax) return n2;
    return bwd_slab(n0, n1, n2);
}
inline size_t bwd_smem(int gpad, int n0, int n1, int n2, int ng, bool x3 = false)
{
    return bwd_smem_slab(gpad, n0, n1, n2, ng, bwd_slab_for(gpad, n0, n1, n2, x3), x3);
}
inline uint32_t pow2cols(int n) { uint32_t c = 32; while ((int)c < n) c <<= 1; return c; }

// CTAs per SM as the driver sees it (registers, threads, shared memory) and TMEM columns (512 per SM).
// The first version of this file modelled shared memory only and believed in 4 CTAs per SM where the
// register file allowed one (profiles/r1_notes.md: the last CTA of SA1 forward started 66 us after the first).
template <class Kern>
int ctas_per_sm(Kern kern, int threads, size_t smem, int tmem_cols)
{
    // one kernel instantiation serves several levels: raise the opt-in limit to the file's maximum once, never lower it
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return 0;
    const size_t dyn_max = (size_t)232448 - fa.sharedSizeBytes;          // 227 KB per CTA, static part included
    if (smem > dyn_max) return 0;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_max) != cudaSuccess) { cudaGetLastError(); return 0; }
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem) != cudaSuccess) return 0;
    occ = occ < 512 / tmem_cols ? occ : 512 / tmem_cols;
    return occ > 8 ? 8 : occ;
}

int num_sms()
{
    if (g_num_sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            g_num_sms = 0;
    }
    return g_num_sms;
}

template <int K> void (*fwd_kern(int ng))(SaFwdArgs)
{
    return ng == 1 ? sa_fwd_kernel<K, 1, false> : ng == 2 ? sa_fwd_kernel<K, 2, false> : ng == 3 ? sa_fwd_kernel<K, 3, false> : sa_fwd_kernel<K, 4, false>;
}
template <int K> void (*bwd_kern(int ng))(SaBwdArgs)
{
    return ng == 1 ? sa_bwd_kernel<K, 1, false> : ng == 2 ? sa_bwd_kernel<K, 2, false> : ng == 3 ? sa_bwd_kernel<K, 3, false> : sa_bwd_kernel<K, 4, false>;
}
// compacted-row variants (the template's K is unused by them: the octet structure replaces it)
void (*fwd_kern_cp(int ng))(SaFwdArgs)
{
    return ng == 1 ? sa_fwd_kernel<32, 1, true> : ng == 2 ? sa_fwd_kernel<32, 2, true> : ng == 3 ? sa_fwd_kernel<32, 3, true> : sa_fwd_kernel<32, 4, true>;
}
void (*fwd_kern_cp_x3(int ng))(SaFwdArgs)
{
    return ng == 1 ? sa_fwd_kernel<32, 1, true, true> : ng == 2 ? sa_fwd_kernel<32, 2, true, true> : ng == 3 ? sa_fwd_kernel<32, 3, true, true> : sa_fwd_kernel<32, 4, true, true>;
}
void (*bwd_kern_cp_x3(int ng))(SaBwdArgs)
{
    return ng == 1 ? sa_bwd_kernel<32, 1, true, true> : ng == 2 ? sa_bwd_kernel<32, 2, true, true> : ng == 3 ? sa_bwd_kernel<32, 3, true, true> : sa_bwd_kernel<32, 4, true, true>;
}
void (*bwd_kern_cp(int ng))(SaBwdArgs)
{
    return ng == 1 ? sa_bwd_kernel<32, 1, true> : ng == 2 ? sa_bwd_kernel<32, 2, true> : ng == 3 ? sa_bwd_kernel<32, 3, true> : sa_bwd_kernel<32, 4, true>;
}

// tiles in flight per SM = NG (per CTA, sharing the resident weights) x CTAs per SM: take the combination
// that keeps the most tiles in flight (the per-tile chain is latency-bound); ties go to the larger NG
// (fewer CTAs: fewer prologues, weights loaded fewer times).  Decisions are cached per configuration.
struct Pick { int ng, occ; };
template <class KernOf, class SmemOf>
Pick pick_ng(KernOf kern_of, SmemOf smem_of, int gc)
{
    Pick best{0, 0};
    int best_tiles = 0;
    for (int ng = 1; ng <= 4; ++ng) {
        const size_t sm = smem_of(ng);
        if (sm > kSmemPerCtaMax || ng * gc > 512) break;
        const int occ = ctas_per_sm(kern_of(ng), ng * 160, sm, (int)pow2cols(ng * gc));
        if (ng * occ >= best_tiles && occ > 0) { best_tiles = ng * occ; best = Pick{ng, occ}; }
    }
    return best;
}

struct PickKey { int dir, K, gpad, n0, n1, n2, dev; };
struct PickEnt { PickKey k; Pick p; };
PickEnt g_picks[128];
int g_npicks = 0;

template <class KernOf, class SmemOf>
Pick cached_pick(int dir, int K, int gpad, int n0, int n1, int n2, KernOf kern_of, SmemOf smem_of, int gc)
{
    // the pick also carries a side effect of ctas_per_sm (the per-device shared-memory opt-in), so it is keyed by device
    int dev = 0;
    cudaGetDevice(&dev);
    const PickKey key{dir, K, gpad, n0, n1, n2, dev};
    for (int i = 0; i < g_npicks; ++i) {
        const PickKey &q = g_picks[i].k;
        if (q.dir == dir && q.K == K && q.gpad == gpad && q.n0 == n0 && q.n1 == n1 && q.n2 == n2 && q.dev == dev) return g_picks[i].p;
    }
    const Pick p = pick_ng(kern_of, smem_of, gc);
    if (g_npicks < 128) g_picks[g_npicks++] = PickEnt{key, p};
    return p;
}
}  // namespace

bool psg_sa_fusable(int K, int gpad, int n0, int n1, int n2)
{
    if (K != 16 && K != 32) return false;
    if (gpad % 16 || n0 % 16 || n1 % 16 || n2 % 16) return false;
    if (gpad > 128 || n0 > 128 || n1 > 128 || n2 > 128) return false;
    return fwd_smem(gpad, n0, n1, n2, 1) <= kSmemPerCtaMax && bwd_smem(gpad, n0, n1, n2, 1) <= kSmemPerCtaMax;
}

// the segmented pool of the compacted-row kernels borrows 4 KB of the tile's operand buffer per warp
bool psg_sa_compactable(int K, int gpad, int n0, int n1, int n2)
{
    return psg_sa_fusable(K, gpad, n0, n1, n2) && fwd_smem(gpad, n0, n1, n2, 1, true) <= kSmemPerCtaMax;
}

// can the branch run as 3xTF32 fused kernels (hi + lo weights and operand buffers in shared memory, one tile in flight)?
bool psg_sa_fusable_x3(int K, int gpad, int n0, int n1, int n2)
{
    if (!psg_sa_compactable(K, gpad, n0, n1, n2)) return false;
    return fwd_smem(gpad, n0, n1, n2, 1, true, true) <= kSmemPerCtaMax && bwd_smem(gpad, n0, n1, n2, 1, true) <= kSmemPerCtaMax;
}

size_t psg_sa_mask_words(long long rows, int n)
{
    return (size_t)((rows + 127) / 128) * ((n + 31) / 32) * 128;
}

int psg_sa_fused_fwd(const PsgSaFused &f, cudaStream_t st)
{
    SaFwdArgs a;
    a.feats = f.feats; a.D = f.D; a.xyz = f.xyz; a.cloud_stride = f.cloud_stride; a.nclouds = f.nclouds; a.Nsrc = f.Nsrc;
    a.new_xyz = f.new_xyz; a.idx = f.idx; a.rows = f.rows; a.S = f.S;
    a.gpad = f.gpad; a.n0 = f.n[0]; a.n1 = f.n[1]; a.n2 = f.n[2];
    a.w0 = f.wf[0]; a.w1 = f.wf[1]; a.w2 = f.wf[2]; a.nw0 = f.nwf[0]; a.nw1 = f.nwf[1]; a.nw2 = f.nwf[2];
    a.b0 = f.bias[0]; a.b1 = f.bias[1]; a.b2 = f.bias[2];
    a.m0 = f.m0; a.m1 = f.m1; a.out = f.out; a.arg = f.arg;
    a.ntiles = (int)((f.rows + 127) / 128);
    a.trace = psg_tile_trace_slot();
    a.crow_src = f.crow_src; a.crow_g = f.crow_g; a.ntiles_dev = f.ntiles_dev;
    a.w0l = f.wf_lo[0]; a.w1l = f.wf_lo[1]; a.w2l = f.wf_lo[2];
    const bool cp = f.crow_src && f.crow_g && f.ntiles_dev;
    const bool x3 = a.w0l && a.w1l && a.w2l;
    const int gc = (int)pow2cols(a.n0 > a.n1 ? (a.n0 > a.n2 ? a.n0 : a.n2) : (a.n1 > a.n2 ? a.n1 : a.n2));
    if (f.K != 16 && f.K != 32) return PSG_EUNSUPPORTED;
    if (cp && !psg_sa_compactable(f.K, a.gpad, a.n0, a.n1, a.n2)) return PSG_EUNSUPPORTED;
    if (x3 && !cp) return PSG_EUNSUPPORTED;
    auto smem_of = [&](int g) { return fwd_smem(a.gpad, a.n0, a.n1, a.n2, g, cp, x3); };
    const Pick pk = x3 ? cached_pick(4, 32, a.gpad, a.n0, a.n1, a.n2, fwd_kern_cp_x3, smem_of, gc)
                  : cp ? cached_pick(2, 32, a.gpad, a.n0, a.n1, a.n2, fwd_kern_cp, smem_of, gc)
                  : f.K == 32 ? cached_pick(0, 32, a.gpad, a.n0, a.n1, a.n2, fwd_kern<32>, smem_of, gc)
                              : cached_pick(0, 16, a.gpad, a.n0, a.n1, a.n2, fwd_kern<16>, smem_of, gc);
    if (pk.ng < 1 || pk.occ < 1 || num_sms() < 1) return PSG_EUNSUPPORTED;
    // compacted rows: only the device knows the tile count; the persistent CTAs stride over whatever there is.  The grid
    // is sized for the padded tiles (CTAs without a tile leave after the prologue): a grid for an S3DIS-density guess of
    // rows / 3 left SA2 (rows / 2, not / 3.6) on 86 of 148 SMs for two rounds of tiles
    const int want = (a.ntiles + pk.ng - 1) / pk.ng, cap = num_sms() * pk.occ;
    const int grid = want < cap ? want : cap;
    auto kern = x3 ? fwd_kern_cp_x3(pk.ng) : cp ? fwd_kern_cp(pk.ng) : f.K == 32 ? fwd_kern<32>(pk.ng) : fwd_kern<16>(pk.ng);
    { cudaError_t e__ = psg_launch_pdl(kern, dim3(grid), dim3(pk.ng * 160), smem_of(pk.ng), st, 1, a);
      if (e__ != cudaSuccess) { fprintf(stderr, "sa launch: %s (ng %d occ %d grid %d smem %zu)\n", cudaGetErrorString(e__), pk.ng, pk.occ, grid, smem_of(pk.ng)); return PSG_ECUDA; } }
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

int psg_sa_fused_bwd(const PsgSaFused &f, TView dout, TView dG, int gcols, float *dG_rm, int rm_only, cudaStream_t st)
{
    SaBwdArgs a;
    a.dout = dout; a.outv = f.out; a.arg = f.arg; a.m0 = f.m0; a.m1 = f.m1;
    a.wb0 = f.wb[0]; a.wb1 = f.wb[1]; a.wb2 = f.wb[2]; a.nwb0 = f.nwb[0]; a.nwb1 = f.nwb[1]; a.nwb2 = f.nwb[2];
    a.dG = dG; a.gcols = gcols; a.rows = f.rows;
    a.dG_rm = dG_rm; a.rm_only = (dG_rm && rm_only) ? 1 : 0;
    a.wb0l = f.wb_lo[0]; a.wb1l = f.wb_lo[1]; a.wb2l = f.wb_lo[2];
    const bool x3 = a.wb0l && a.wb1l && a.wb2l;
    a.slab = bwd_slab_for(f.gpad, f.n[0], f.n[1], f.n[2], x3);
    a.gpad = f.gpad; a.n0 = f.n[0]; a.n1 = f.n[1]; a.n2 = f.n[2];
    a.ntiles = (int)((f.rows + 127) / 128);
    a.trace = psg_tile_trace_slot();
    a.crow_g = f.crow_g; a.ntiles_dev = f.ntiles_dev;
    const bool cp = f.crow_src && f.crow_g && f.ntiles_dev;
    if (x3 && !cp) return PSG_EUNSUPPORTED;
    const int gc = (int)pow2cols(a.n0 > a.n1 ? (a.n0 > a.gpad ? a.n0 : a.gpad) : (a.n1 > a.gpad ? a.n1 : a.gpad));
    if (f.K != 16 && f.K != 32) return PSG_EUNSUPPORTED;
    auto smem_of = [&](int g) { return bwd_smem(a.gpad, a.n0, a.n1, a.n2, g, x3); };
    const Pick pk = x3 ? cached_pick(5, 32, a.gpad, a.n0, a.n1, a.n2, bwd_kern_cp_x3, smem_of, gc)
                  : cp ? cached_pick(3, 32, a.gpad, a.n0, a.n1, a.n2, bwd_kern_cp, smem_of, gc)
                  : f.K == 32 ? cached_pick(1, 32, a.gpad, a.n0, a.n1, a.n2, bwd_kern<32>, smem_of, gc)
                              : cached_pick(1, 16, a.gpad, a.n0, a.n1, a.n2, bwd_kern<16>, smem_of, gc);
    if (pk.ng < 1 || pk.occ < 1 || num_sms() < 1) return PSG_EUNSUPPORTED;
    const int want = (a.ntiles + pk.ng - 1) / pk.ng, cap = num_sms() * pk.occ;
    const int grid = want < cap ? want : cap;
    auto kern = x3 ? bwd_kern_cp_x3(pk.ng) : cp ? bwd_kern_cp(pk.ng) : f.K == 32 ? bwd_kern<32>(pk.ng) : bwd_kern<16>(pk.ng);
    { cudaError_t e__ = psg_launch_pdl(kern, dim3(grid), dim3(pk.ng * 160), smem_of(pk.ng), st, 1, a);
      if (e__ != cudaSuccess) { fprintf(stderr, "sa launch: %s (ng %d occ %d grid %d smem %zu)\n", cudaGetErrorString(e__), pk.ng, pk.occ, grid, smem_of(pk.ng)); return PSG_ECUDA; } }
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
