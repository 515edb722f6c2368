// chain_fused.cu -- "tile programs": chains of row-local layers executed per 128-row tile entirely
// on-chip (tcgen05 TF32, TMEM accumulator, activations in one shared-memory A-operand buffer that
// every layer overwrites in place), with the weights streamed through a TMA ring.
//
// One kernel, driven by a small op list built on the host, covers
//   * fp1 + head forward [+ loss gradient + backward]       (psg_chain_fused)
//   * wide set-abstraction levels, forward and backward     (psg_sa_stream_fwd / _bwd)
//   * feature-propagation levels, forward and backward      (psg_fp_stream_fwd / _bwd)
// i.e. every place where the reference runs conv1x1 + BN + ReLU chains whose weights do not fit
// in shared memory next to the activations (the narrow SA levels keep their weights resident:
// sa_fused.cu).
//
// Reference: PointNet/models/pointnet_util.py:126-137,200-205 (group + MLP + max), :305-319
// (interpolate + concat + MLP), pointnet2_sem_seg.py:34-39 (fp1, conv1, bn1, conv2, log_softmax), the
// attack costs of nontarget.py:34,120-128 / target.py:38,149-168, and autograd of all of it.
//
// Roles per CTA: NG x 4 worker warps (thread = tile row = TMEM lane; they fill the A operand --
// gather / interpolate / scatter / load -- and run the epilogues), one MMA-issuing thread, one
// weight-producer thread.  A weight stage is consumed by all NG tiles in flight before it is
// released, so the L2 -> SM weight traffic is shared between them.
#include "psg_common.cuh"
#include "psg_internal.h"
#include "psg_loss.cuh"
#include "psg_tc.cuh"
#include "psg_epi.cuh"

long long *psg_tile_trace_slot();

namespace {

constexpr int kWorkers = 128;
constexpr int kStages = 2;
constexpr int kMaskSlots = 4;
constexpr int kMaxOps = PSG_CHAIN_MAX_OPS;

enum { PRE_NONE = 0, PRE_GROUP, PRE_FP, PRE_LOAD, PRE_SCATTER };
enum { EPI_NONE = 0, EPI_RELU, EPI_MASK, EPI_HEAD, EPI_STORE, EPI_MAXPOOL };

struct TileOp {
    const float *w;            // packed weights [plane][wstride rows][4]
    const float *wlo;          // X3 programs: the TF32 residual of w (same packing), or null
    int wstride, wrow0, wplane0;
    int n, planes;             // MMA N; K / 4
    int aplane0;               // first A-buffer plane read
    int accumulate;            // continue the previous op's accumulator
    int pps;                   // planes per weight stage (even)
    int pre, pre_a;            // A refill before this op (PRE_SCATTER: first column)
    int epi, relu;
    const float *bias;
    int boff;                  // offset of this op's bias copy in the shared-memory bias area (floats)
    int slot;                  // shared-memory mask slot or -1
    unsigned *mglobal;         // global ReLU bits of this op's output [tile][words][128] or null
    TView out;                 // EPI_STORE / EPI_MAXPOOL destination (column offset folded into c0)
    float *rm; int rm_stride;  // EPI_STORE: optional row-major mirror of `out` (floats per row), or null
    int rm_only;               // ... and skip the T-layout store
    TView out2; int out2_cols; // EPI_STORE: columns (absolute, of this op's range) below out2_cols are also written here
    unsigned char *arg; int argC, arg0;   // EPI_MAXPOOL
};

struct TileSrc {
    // PRE_GROUP
    TView feats; int D, gpad; const float *xyz; long long cloud_stride; int nclouds, Nsrc;
    const float *new_xyz; const int *idx; int S, K;
    // PRE_FP: skip rows (row-local) into planes [0, lcols/4), interpolation into planes [iplane0, ...)
    // PRE_LOAD: lsrc rows only
    TView lsrc; int lcols;
    TView isrc; int iS, iNf, icols, iplane0; const int *nn_idx; const float *nn_w;
    const float *irm; int irm_stride;    // row-major mirror of isrc (whole 32-byte sectors per request), or null
    // PRE_SCATTER
    TView dout, outv; const unsigned char *sarg; int sargC;
};

struct TileArgs {
    TileOp ops[kMaxOps];
    int nops;
    TileSrc src;
    long long rows; int ntiles;
    int abytes, stage_bytes, tcols;      // A buffer bytes per tile, weight stage bytes, TMEM columns per tile
    int rmstage;                         // 1: a 4 KB per-warp staging area for coalesced row-major stores follows the scatter staging
    int acols;                           // TS programs: TMEM columns of the A operand (after the accumulator's tcols)
    int lo_off;                          // X3 programs: operand column where the A_lo copy of the operand starts
    int bias_floats;                     // size of the shared-memory bias area
    int mwords, mbytes;                  // ReLU-bit words per mask slot; bytes of the per-tile mask / scratch area
    // head / loss (EPI_HEAD)
    int backward, ncls, loss_kind, target;
    const int *labels; float scale, kappa; const float *dlogp;
    float *loss_rows; unsigned char *hit;
    TView zout;
    long long *trace;                    // debug: clock64 stamps of CTA 0 ([role][512]; psg_debug_trace), or null
};

__device__ __forceinline__ float4 *plane_ptr(unsigned char *buf, int chunk, int row)
{
    return reinterpret_cast<float4 *>(buf) + (size_t)chunk * 128 + row;
}
__device__ __forceinline__ uint32_t pow2cols_dev(uint32_t n) { uint32_t c = 32; while (c < n) c <<= 1; return c; }

// ---- A-operand producers (worker thread r owns tile row r) ----------------------------------------
__device__ __forceinline__ void pre_group(const TileSrc &s, unsigned char *pA, long long row, bool valid, int r)
{
    const long long rr = valid ? row : 0;
    const long long ps = rr / s.K;
    const int p = (int)(ps / s.S);
    const int src = s.idx[rr];
    const int cloud = p % s.nclouds;
    const long long srow = (long long)cloud * s.Nsrc + src;
    const int D = s.D, nfull = D >> 2;
    {
        const float *fb = s.feats.base + tv_off(s.feats, srow, 0);
        constexpr int NB = 16;                       // independent 16-byte requests in flight per thread
        for (int c0 = 0; c0 < nfull; c0 += NB) {
            float4 x[NB];
#pragma unroll
            for (int j = 0; j < NB; ++j)
                x[j] = c0 + j < nfull ? __ldg(reinterpret_cast<const float4 *>(fb + (size_t)(c0 + j) * 512)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < NB; ++j)
                if (c0 + j < nfull) *plane_ptr(pA, c0 + j, r) = valid ? x[j] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    const float *sp = s.xyz + (long long)cloud * s.cloud_stride + (long long)src * 3;
    const float *cp = s.new_xyz + ps * 3;
    const float dx = __fsub_rn(sp[0], cp[0]), dy = __fsub_rn(sp[1], cp[1]), dz = __fsub_rn(sp[2], cp[2]);
    for (int c = nfull; c < s.gpad / 4; ++c) {
        float f[4] = {0.f, 0.f, 0.f, 0.f};
        if (4 * c < D) { float4 q = tv_ld(s.feats, srow, c); f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w; }
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ch = 4 * c + j;
            o[j] = ch < D ? f[j] : (ch == D ? dx : (ch == D + 1 ? dy : (ch == D + 2 ? dz : 0.f)));
            if (!valid) o[j] = 0.f;
        }
        *plane_ptr(pA, c, r) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// source chunks [cbeg, cbeg + nch) of the row-local tensor -> A planes [0, nch)
__device__ __forceinline__ void pre_load(const TileSrc &s, unsigned char *pA, long long row, bool valid, int r, int cbeg, int nch)
{
    const float *b = s.lsrc.base + tv_off(s.lsrc, valid ? row : 0, cbeg);
    constexpr int NB = 16;
    for (int c0 = 0; c0 < nch; c0 += NB) {
        float4 x[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j)
            x[j] = c0 + j < nch ? *reinterpret_cast<const float4 *>(b + (size_t)(c0 + j) * 512) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < NB; ++j)
            if (c0 + j < nch) *plane_ptr(pA, c0 + j, r) = valid ? x[j] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// (f[i0] w0 + f[i1] w1) + f[i2] w2, products rounded separately as torch does (pointnet_util.py:308).
// The three gathered rows are 16-byte pieces 2 KB apart: a latency-bound gather, so the loads of eight chunks
// (24 independent 16-byte requests per thread) are issued before the first one is consumed.
// interpolated chunks [cbeg, cbeg + nch) -> A planes [plane0, plane0 + nch)
// TS: the A operand lives in tensor memory (tA = TMEM address of this thread's lane, column 0 of the operand):
// eight chunks are collected and written with one tcgen05.st (nch must then be a multiple of 8)
// X3 (TS only): the operand is written twice -- as it is (the hardware reads its top 19 bits: A_hi) and its residual
// A_lo = A - A_hi at column lo_off
__device__ __forceinline__ void lo32(const float *v, float *l)
{
#pragma unroll
    for (int i = 0; i < 32; ++i) l[i] = v[i] - __uint_as_float(__float_as_uint(v[i]) & 0xFFFFE000u);
}
template <bool TS, bool X3 = false>
__device__ __forceinline__ void pre_interp(const TileSrc &s, unsigned char *pA, long long row, bool valid, int r, int cbeg, int nch,
                                           int plane0, uint32_t tA, int lo_off = 0)
{
    const long long rr = valid ? row : 0;
    const long long p = rr / s.iNf;
    const int *ii = s.nn_idx + rr * 3;
    const float *ww = s.nn_w + rr * 3;
    const long long r0 = p * s.iS + ii[0], r1 = p * s.iS + ii[1], r2 = p * s.iS + ii[2];
    const float w0 = valid ? ww[0] : 0.f, w1 = valid ? ww[1] : 0.f, w2 = valid ? ww[2] : 0.f;
    if (s.irm) {
        // row-major mirror: one 32-byte request per two chunks -- half the L1 tag work and only whole sectors
        // from L2 (the T-layout pieces are 16 bytes, 2 KB apart)
        const float *m0 = s.irm + r0 * s.irm_stride + 4 * cbeg, *m1 = s.irm + r1 * s.irm_stride + 4 * cbeg,
                    *m2 = s.irm + r2 * s.irm_stride + 4 * cbeg;
        constexpr int NP = 4;                         // pairs of chunks per batch
        for (int c0 = 0; c0 < nch; c0 += 2 * NP) {
            float4 x[2 * NP], y[2 * NP], z[2 * NP];
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                const bool in = c0 + 2 * j < nch;
                const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
                x[2 * j] = x[2 * j + 1] = y[2 * j] = y[2 * j + 1] = z[2 * j] = z[2 * j + 1] = zero;
                if (in) {
                    tc::ldg256(m0 + (size_t)(c0 + 2 * j) * 4, x[2 * j], x[2 * j + 1]);
                    tc::ldg256(m1 + (size_t)(c0 + 2 * j) * 4, y[2 * j], y[2 * j + 1]);
                    tc::ldg256(m2 + (size_t)(c0 + 2 * j) * 4, z[2 * j], z[2 * j + 1]);
                }
            }
            float v[8 * NP];
#pragma unroll
            for (int j = 0; j < 2 * NP; ++j) {
                float4 q;
                q.x = __fadd_rn(__fadd_rn(__fmul_rn(x[j].x, w0), __fmul_rn(y[j].x, w1)), __fmul_rn(z[j].x, w2));
                q.y = __fadd_rn(__fadd_rn(__fmul_rn(x[j].y, w0), __fmul_rn(y[j].y, w1)), __fmul_rn(z[j].y, w2));
                q.z = __fadd_rn(__fadd_rn(__fmul_rn(x[j].z, w0), __fmul_rn(y[j].z, w1)), __fmul_rn(z[j].z, w2));
                q.w = __fadd_rn(__fadd_rn(__fmul_rn(x[j].w, w0), __fmul_rn(y[j].w, w1)), __fmul_rn(z[j].w, w2));
                if (TS) { v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w; }
                else if (c0 + j < nch) *plane_ptr(pA, plane0 + c0 + j, r) = q;
            }
            if (TS) tc::tmem_st32(tA + (uint32_t)(plane0 + c0) * 4u, v);
            if (TS && X3) { float l[32]; lo32(v, l); tc::tmem_st32(tA + (uint32_t)(plane0 + c0) * 4u + (uint32_t)lo_off, l); }
        }
        return;
    }
    const float *b0 = s.isrc.base + tv_off(s.isrc, r0, cbeg), *b1 = s.isrc.base + tv_off(s.isrc, r1, cbeg),
                *b2 = s.isrc.base + tv_off(s.isrc, r2, cbeg);
    constexpr int NB = 8;
    for (int c0 = 0; c0 < nch; c0 += NB) {
        float4 x[NB], y[NB], z[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            // (every element is written on every path: a conditional assignment would carry the previous
            // batch's registers around the loop)
            const bool in = c0 + j < nch;
            const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
            x[j] = in ? __ldg(reinterpret_cast<const float4 *>(b0 + (size_t)(c0 + j) * 512)) : zero;
            y[j] = in ? __ldg(reinterpret_cast<const float4 *>(b1 + (size_t)(c0 + j) * 512)) : zero;
            z[j] = in ? __ldg(reinterpret_cast<const float4 *>(b2 + (size_t)(c0 + j) * 512)) : zero;
        }
        float v[4 * NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            float4 q;
            q.x = __fadd_rn(__fadd_rn(__fmul_rn(x[j].x, w0), __fmul_rn(y[j].x, w1)), __fmul_rn(z[j].x, w2));
            q.y = __fadd_rn(__fadd_rn(__fmul_rn(x[j].y, w0), __fmul_rn(y[j].y, w1)), __fmul_rn(z[j].y, w2));
            q.z = __fadd_rn(__fadd_rn(__fmul_rn(x[j].z, w0), __fmul_rn(y[j].z, w1)), __fmul_rn(z[j].z, w2));
            q.w = __fadd_rn(__fadd_rn(__fmul_rn(x[j].w, w0), __fmul_rn(y[j].w, w1)), __fmul_rn(z[j].w, w2));
            if (TS) { v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w; }
            else if (c0 + j < nch) *plane_ptr(pA, plane0 + c0 + j, r) = q;
        }
        if (TS) tc::tmem_st32(tA + (uint32_t)(plane0 + c0) * 4u, v);
        if (TS && X3) { float l[32]; lo32(v, l); tc::tmem_st32(tA + (uint32_t)(plane0 + c0) * 4u + (uint32_t)lo_off, l); }
    }
}

// dY[(g,k)][c] = (k == arg[g][c] && out[g][c] > 0) ? dOut[g][c] : 0 for columns [col0, col0 + 4*planes): the warp fetches
// each chunk of its neighbourhoods once and shares it through a staging area (psg_scatter_warp, psg_epi.cuh)
__device__ __forceinline__ void pre_scatter(const TileSrc &s, unsigned char *pA, long long row, bool valid, int r, int col0,
                                            int planes, float4 *stage_d, uchar4 *stage_a)
{
    const long long g = (valid ? row : 0) / s.K;
    const int lane = r & 31;
    auto put = [&](int c, float4 q) { *plane_ptr(pA, c, r) = q; };
    if (s.K == 32) psg_scatter_warp<32>(s.dout, s.outv, s.sarg, s.sargC, g, valid, lane, col0 >> 2, planes, stage_d, stage_a, put);
    else psg_scatter_warp<16>(s.dout, s.outv, s.sarg, s.sargC, g, valid, lane, col0 >> 2, planes, stage_d, stage_a, put);
}

// CS > 1: a cluster of CS CTAs works on ONE tile (NG == 1); CTA q computes columns [q n/CS, (q+1) n/CS)
// of every layer from the full A operand (replicated in each CTA), streams only its slice of the
// weights, and its epilogue writes its activation slice into every CTA's A buffer through distributed
// shared memory.  Synchronisation stays on mbarriers: the MMA commit is multicast to all CTAs'
// accumulator barriers (nobody overwrites an operand a peer's MMA still reads) and the workers arrive
// on all CTAs' operand barriers (nobody issues an MMA before every slice landed).  This is what lets
// the deep levels -- few rows, large weights -- use more than one SM per tile.
// TS: the A operand of every MMA lives in TENSOR MEMORY (tcgen05.mma with A from TMEM): gathers and epilogues
// write the next operand with tcgen05.st, there is no operand buffer in shared memory at all.  That removes
// the two biggest shared-memory streams of a layer (MMA A reads, epilogue stores) -- the SS-mode chain was
// shared-memory bound at about twice its tensor time -- and leaves room for 64 KB weight stages.
// X3: error-compensated 3xTF32 (TS programs, one tile in flight): every GEMM op runs three passes over its K range --
// A_lo W_hi, A_hi W_lo, A_hi W_hi -- into the same accumulator; the producer streams W_hi, W_lo, W_hi again, the workers
// write every operand twice (A and, at column lo_off, A_lo).  One hand-off per op, as in the plain program.
template <int NG, int CS, bool TS, bool X3 = false>
__global__ void __launch_bounds__(NG * 128 + 64, 1) tile_kernel(const __grid_constant__ TileArgs a)
{
    static_assert(CS == 1 || NG == 1, "cluster programs keep one tile in flight");
    static_assert(!TS || CS == 1, "peers cannot write each other's tensor memory");
    static_assert(!X3 || (TS && NG == 1), "3xTF32 programs keep the operand and its residual in tensor memory");
    // no-swizzle UMMA operands and bulk copies need 16-byte alignment only: a 128-byte aligned dynamic
    // segment keeps the static + padding overhead small (every KB decides whether 32 KB weight stages fit)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar_in[NG], bar_acc[NG], bar_full[kStages], bar_empty[kStages];
    __shared__ uint32_t tmem_slot;

    const uint32_t s0 = tc::smem_u32(smem_raw);
    const uint32_t sbase = (s0 + 127u) & ~127u;
    unsigned char *base = smem_raw + (sbase - s0);
    // [A tile 0 .. NG-1][W stage 0][W stage 1][mask bits tile 0 .. NG-1]
    const uint32_t sA0 = sbase, sW = sbase + NG * a.abytes;
    unsigned char *pA0 = base;
    unsigned *pMask = reinterpret_cast<unsigned *>(base + (size_t)NG * a.abytes + (size_t)kStages * a.stage_bytes);
    float *sbias = reinterpret_cast<float *>(pMask + (size_t)NG * (a.mbytes / 4));
    float4 *stage_d = reinterpret_cast<float4 *>(sbias + a.bias_floats);          // [NG * 4 warps][32]
    uchar4 *stage_a = reinterpret_cast<uchar4 *>(stage_d + NG * 4 * 32);           // [NG * 4 warps][32]
    float4 *stage_rm = reinterpret_cast<float4 *>(stage_a + NG * 4 * 32);          // [NG * 4 warps][256] when a.rmstage

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tper = (uint32_t)(TS ? a.tcols + a.acols : a.tcols);      // TMEM columns per tile in flight
    const uint32_t ncols = pow2cols_dev(tper * NG);
    if (threadIdx.x == 0) {
        for (int g = 0; g < NG; ++g) { tc::mbar_init(tc::smem_u32(&bar_in[g]), kWorkers * CS); tc::mbar_init(tc::smem_u32(&bar_acc[g]), CS); }
        for (int s = 0; s < kStages; ++s) { tc::mbar_init(tc::smem_u32(&bar_full[s]), 1); tc::mbar_init(tc::smem_u32(&bar_empty[s]), 1); }
        tc::fence_mbar_init();
    }
    if (warp == NG * 4) tc::tmem_alloc(tc::smem_u32(&tmem_slot), ncols);
    // biases are constants of the network (not produced by the previous kernel): staged into shared memory
    // here, ahead of griddepcontrol.wait, so no epilogue ever waits on a global load for them
    for (int o = 0; o < a.nops; ++o) {
        const TileOp &op = a.ops[o];
        if (op.bias)
            for (int i = threadIdx.x; i < op.n; i += NG * 128 + 64) sbias[op.boff + i] = __ldg(op.bias + i);
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (CS > 1) tc::cluster_sync_all();            // peers' barriers exist before anyone arrives on them remotely
    tc::pdl_launch_dependents();
    // everything above overlapped the previous kernel's tail.  The weight producer does not wait at all: it reads only
    // the network's constant weights, so its first stages land while the predecessor is still draining.
    if (warp != NG * 4 + 1) tc::pdl_wait();
    const uint32_t tmem = tmem_slot;
    const int q = CS > 1 ? (int)tc::cluster_ctarank() : 0;
    const int first_tile = (CS > 1 ? (int)blockIdx.x / CS : (int)blockIdx.x) * NG;
    const int tstride = (CS > 1 ? (int)gridDim.x / CS : (int)gridDim.x) * NG;

    if (warp == NG * 4 + 1) {
        // ---------------- weight producer: the whole warp issues a stage's copies ----------------
        // (column-sliced weights are one copy per 4-column plane; a single thread issuing them back to back cost
        // ~80 ns per copy -- 1.3 us per 32 KB stage of a cluster program, more than the copies take to arrive)
        int it = 0;
        for (int tile0 = first_tile; tile0 < a.ntiles; tile0 += tstride) {
            for (int o = 0; o < a.nops; ++o) {
                const TileOp &op = a.ops[o];
                const int nl = op.n / CS;                     // this CTA's slice of the output columns
                const int nsub = (X3 && op.wlo) ? 3 : 1;
                for (int sub = 0; sub < nsub; ++sub)
                for (int pl = 0; pl < op.planes; pl += op.pps, ++it) {
                    const int np = min(op.pps, op.planes - pl);
                    const int slot = it % kStages;
                    const uint32_t ph = (uint32_t)(it / kStages) & 1u;
                    const uint32_t full = tc::smem_u32(&bar_full[slot]);
                    const uint32_t dst = sW + slot * a.stage_bytes;
                    if (lane == 0) {
                        tc::mbar_spin(tc::smem_u32(&bar_empty[slot]), ph ^ 1u);
                        tc::mbar_expect_tx(full, (uint32_t)np * nl * 16);
                    }
                    __syncwarp();
                    const float4 *wsrc = reinterpret_cast<const float4 *>((X3 && sub == 1) ? op.wlo : op.w) + (size_t)(op.wplane0 + pl) * op.wstride +
                                         op.wrow0 + q * nl;
                    if (op.wstride == nl) {
                        if (lane == 0) tc::bulk_g2s(dst, wsrc, (uint32_t)np * nl * 16, full);
                    } else {
                        for (int j = lane; j < np; j += 32)
                            tc::bulk_g2s(dst + j * nl * 16, wsrc + (size_t)j * op.wstride, (uint32_t)nl * 16, full);
                    }
                }
            }
        }
    } else if (warp == NG * 4) {
        // ---------------- MMA issuer ----------------
        if (lane == 0) {
            int it = 0;
            long long *tr = (a.trace && blockIdx.x == 0) ? a.trace + 2 * 512 : nullptr;
            int tn = 0;
            uint32_t ph_in[NG];
#pragma unroll
            for (int g = 0; g < NG; ++g) ph_in[g] = 0u;
            for (int tile0 = first_tile; tile0 < a.ntiles; tile0 += tstride) {
                for (int o = 0; o < a.nops; ++o) {
                    const TileOp &op = a.ops[o];
                    const int nl = op.n / CS;
                    const uint32_t idesc = tc::idesc_tf32(128, nl);
                    const int nst = (op.planes + op.pps - 1) / op.pps;
                    if (NG == 2 && nst <= kStages) {
                        // Tile-major order (the whole op fits in the ring): tile 0's accumulator completes after
                        // ITS MMAs only, so its epilogue overlaps tile 1's MMAs and vice versa on the next op.
                        const int glast = (tile0 + 1 < a.ntiles) ? 1 : 0;
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            if (g > glast) continue;
                            tc::mbar_spin(tc::smem_u32(&bar_in[g]), ph_in[g]); ph_in[g] ^= 1u;
                            if (tr && tn < 510) tr[tn++] = clock64();
                            for (int si = 0; si < nst; ++si) {
                                const int pl = si * op.pps;
                                const int np = min(op.pps, op.planes - pl);
                                const int slot = (it + si) % kStages;
                                if (g == 0) tc::mbar_spin(tc::smem_u32(&bar_full[slot]), (uint32_t)((it + si) / kStages) & 1u);
                                tc::fence_after_sync();
                                const uint32_t sA = sA0 + g * a.abytes + (uint32_t)(op.aplane0 + pl) * 2048u;
                                const uint32_t sB = sW + slot * a.stage_bytes;
                                const uint32_t tD = tmem + g * tper, tA = tD + a.tcols + (uint32_t)(op.aplane0 + pl) * 4u;
                                for (int j = 0; j < np; j += 2) {
                                    const uint64_t bd = tc::smem_desc(sB + j * nl * 16, (uint32_t)(nl * 16), 128);
                                    const uint32_t acc = (op.accumulate || pl > 0 || j > 0) ? 1u : 0u;
                                    if (TS) tc::mma_tf32_ts(tD, tA + j * 4, bd, idesc, acc);
                                    else tc::mma_tf32(tD, tc::smem_desc(sA + j * 2048, 2048, 128), bd, idesc, acc);
                                }
                                if (g == glast) tc::mma_commit(tc::smem_u32(&bar_empty[slot]));
                            }
                            tc::mma_commit(tc::smem_u32(&bar_acc[g]));
                            if (tr && tn < 510) tr[tn++] = clock64();
                        }
                        it += nst;
                        continue;
                    }
                    const int nsub = (X3 && op.wlo) ? 3 : 1;
                    for (int sub = 0; sub < nsub; ++sub)
                    for (int pl = 0; pl < op.planes; pl += op.pps, ++it) {
                        const int np = min(op.pps, op.planes - pl);
                        const int slot = it % kStages;
                        const bool last = pl + op.pps >= op.planes && sub == nsub - 1;
                        tc::mbar_spin(tc::smem_u32(&bar_full[slot]), (uint32_t)(it / kStages) & 1u);
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            if (tile0 + g >= a.ntiles) continue;
                            if (pl == 0 && sub == 0) {
                                // (cluster programs too: what the peers' arrivals publish is SHARED memory -- their operand
                                // slices in this CTA's buffer -- so a CTA-scope acquire orders everything that is read next.
                                // The cluster-scope form makes the compiler invalidate the whole L1 after every wait
                                // (CCTL.IVALL: a quarter of SA4's stall samples, profiles/r2_notes.md))
                                tc::mbar_spin(tc::smem_u32(&bar_in[g]), ph_in[g]);
                                ph_in[g] ^= 1u;
                            }
                            tc::fence_after_sync();
                            const uint32_t sA = sA0 + g * a.abytes + (uint32_t)(op.aplane0 + pl) * 2048u;
                            const uint32_t sB = sW + slot * a.stage_bytes;
                            // X3: the first pass contracts A_lo (operand column lo_off) with W_hi, then A with W_lo, then A with W_hi
                            const uint32_t tD = tmem + g * tper,
                                           tA = tD + a.tcols + (uint32_t)(op.aplane0 + pl) * 4u + ((X3 && nsub == 3 && sub == 0) ? (uint32_t)a.lo_off : 0u);
                            for (int j = 0; j < np; j += 2) {
                                const uint64_t bd = tc::smem_desc(sB + j * nl * 16, (uint32_t)(nl * 16), 128);
                                const uint32_t acc = (op.accumulate || pl > 0 || j > 0 || sub > 0) ? 1u : 0u;
                                if (TS) tc::mma_tf32_ts(tD, tA + j * 4, bd, idesc, acc);
                                else tc::mma_tf32(tD, tc::smem_desc(sA + j * 2048, 2048, 128), bd, idesc, acc);
                            }
                            if (last) {
                                if (CS > 1) tc::mma_commit_mc(tc::smem_u32(&bar_acc[g]), (uint16_t)((1u << CS) - 1u));
                                else tc::mma_commit(tc::smem_u32(&bar_acc[g]));
                            }
                        }
                        tc::mma_commit(tc::smem_u32(&bar_empty[slot]));     // stage free once every tile consumed it
                    }
                }
            }
        }
    } else {
        // ---------------- workers ----------------
        const int grp = warp >> 2, wq = warp & 3;
        const int r = threadIdx.x & 127;
        unsigned char *pA = pA0 + (size_t)grp * a.abytes;
        unsigned *mbits = pMask + (size_t)grp * (a.mbytes / 4);
        const int mw = a.mwords;
        const uint32_t b_in = tc::smem_u32(&bar_in[grp]), b_acc = tc::smem_u32(&bar_acc[grp]);
        const uint32_t tl = tmem + grp * tper + ((uint32_t)(wq * 32) << 16);
        const uint32_t tla = tl + a.tcols;                 // TS: this thread's lane of the A operand
        const int K = a.src.K > 0 ? a.src.K : 32;
        uint32_t ph = 0;
        long long *tr = (a.trace && blockIdx.x == 0 && r == 0) ? a.trace + grp * 512 : nullptr;
        int tn = 0;
        // write 16 bytes of the A operand here and, in a cluster, at the same place in every peer CTA
        auto put = [&](int chunk, float4 val) {
            float4 *dstp = plane_ptr(pA, chunk, r);
            *dstp = val;
            if (CS > 1) {
                const uint32_t la = tc::smem_u32(dstp);
#pragma unroll
                for (int pr = 0; pr < CS; ++pr)
                    if (pr != q) tc::st_cluster_v4(tc::mapa(la, (uint32_t)pr), val);
            }
        };
        // 32 / 16 consecutive columns of this thread's row, starting at operand column `col`
        auto put32 = [&](int col, const float *v) {
            if (TS) {
                tc::tmem_st32(tla + (uint32_t)col, v);
                if (X3) { float l[32]; lo32(v, l); tc::tmem_st32(tla + (uint32_t)(col + a.lo_off), l); }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) put((col >> 2) + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
            }
        };
        auto put16 = [&](int col, const float *v) {
            if (TS) {
                tc::tmem_st16(tla + (uint32_t)col, v);
                if (X3) {
                    float l[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) l[i] = v[i] - __uint_as_float(__float_as_uint(v[i]) & 0xFFFFE000u);
                    tc::tmem_st16(tla + (uint32_t)(col + a.lo_off), l);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) put((col >> 2) + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
            }
        };
        for (int tile = first_tile + grp; tile < a.ntiles; tile += tstride) {
            const long long row = (long long)tile * 128 + r;
            const bool valid = row < a.rows;
            for (int o = 0; o < a.nops; ++o) {
                const TileOp &op = a.ops[o];
                const int nl = op.n / CS, c0l = q * nl;        // this CTA's output columns [c0l, c0l + nl)
                // ---- refill the A operand, hand it to the MMA thread ----
                if (op.pre == PRE_GROUP) pre_group(a.src, pA, row, valid, r);
                else if (op.pre == PRE_FP) {
                    // chunks [pre_a, pre_a + planes) of the concatenation [skip | interpolation]
                    const int L = a.src.lcols / 4, kb = op.pre_a, ke = op.pre_a + op.planes;
                    if (kb < L) pre_load(a.src, pA, row, valid, r, kb, min(ke, L) - kb);
                    if (ke > L) pre_interp<TS, X3>(a.src, pA, row, valid, r, max(kb, L) - L, ke - max(kb, L), max(kb, L) - kb, tla, a.lo_off);
                }
                else if (op.pre == PRE_LOAD) pre_load(a.src, pA, row, valid, r, 0, a.src.lcols / 4);
                else if (op.pre == PRE_SCATTER) pre_scatter(a.src, pA, row, valid, r, op.pre_a, op.planes, stage_d + warp * 32, stage_a + warp * 32);
                tc::fence_before_sync();
                if (CS > 1) {
                    tc::fence_async_all();
                    tc::fence_release_cluster();
#pragma unroll
                    for (int pr = 0; pr < CS; ++pr) tc::mbar_arrive_cluster_relaxed(tc::mapa(b_in, (uint32_t)pr));
                } else {
                    if (TS) tc::tmem_wait_st();        // the operand written by this thread (gather or previous epilogue) has landed
                    else tc::fence_async_smem();
                    tc::mbar_arrive(b_in);
                }
                if (tr && tn < 510) tr[tn++] = clock64();
                // ---- epilogue ----
                tc::mbar_wait(b_acc, ph);          // (CTA-scope acquire in cluster programs as well: see the issuer's wait)
                ph ^= 1u; tc::fence_after_sync();
                if (tr && tn < 510) tr[tn++] = clock64();
                const int words = (op.n + 31) / 32;
                const int w0l = c0l >> 5;
                if (op.epi == EPI_RELU) {
                    int c = 0;
                    for (; c + 32 <= nl; c += 32) {
                        float v[32];
                        tc::tmem_ld32(tl + (uint32_t)c, v);
                        const unsigned w = psg_relu_bias_bits<32>(v, sbias + op.boff + c0l + c);
                        put32(c0l + c, v);
                        if (op.slot >= 0) mbits[((size_t)op.slot * mw + w0l + (c >> 5)) * 128 + r] = w;
                        if (op.mglobal) op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r] = w;
                    }
                    if (c < nl) {
                        float v[16];
                        tc::tmem_ld16(tl + (uint32_t)c, v);
                        const unsigned w = psg_relu_bias_bits<16>(v, sbias + op.boff + c0l + c);
                        put16(c0l + c, v);
                        if (op.slot >= 0) mbits[((size_t)op.slot * mw + w0l + (c >> 5)) * 128 + r] = w;
                        if (op.mglobal) op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r] = w;
                    }
                } else if (op.epi == EPI_MASK) {
                    int c = 0;
                    for (; c + 32 <= nl; c += 32) {
                        const unsigned w = op.mglobal ? op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r]
                                                      : mbits[((size_t)op.slot * mw + w0l + (c >> 5)) * 128 + r];
                        float v[32];
                        tc::tmem_ld32(tl + (uint32_t)c, v);
                        psg_apply_bits<32>(v, w);
                        put32(c0l + c, v);
                    }
                    if (c < nl) {
                        const unsigned w = op.mglobal ? op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r]
                                                      : mbits[((size_t)op.slot * mw + w0l + (c >> 5)) * 128 + r];
                        float v[16];
                        tc::tmem_ld16(tl + (uint32_t)c, v);
                        psg_apply_bits<16>(v, w);
                        put16(c0l + c, v);
                    }
                } else if (op.epi == EPI_STORE) {
                    int c = 0;
                    for (; c + 32 <= nl; c += 32) {
                        float v[32];
                        tc::tmem_ld32(tl + (uint32_t)c, v);
                        unsigned w = 0;
                        if (op.relu) w = psg_relu_bias_bits<32>(v, sbias + op.boff + c0l + c);
                        if (valid) {
                            if (!op.rm_only) {
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    tv_st(op.out, row, ((c0l + c) >> 2) + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
                            }
                            if (op.rm && !a.rmstage) {
                                float4 *d = reinterpret_cast<float4 *>(op.rm + row * op.rm_stride + c0l + c);
#pragma unroll
                                for (int j = 0; j < 8; ++j) d[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                            }
                        }
                        if (valid && op.out2.base && c0l + c + 32 <= op.out2_cols) {
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                tv_st(op.out2, row, ((c0l + c) >> 2) + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
                        }
                        if (op.rm && a.rmstage) {             // whole warp: coalesced row-major store through the staging area
                            const long long row0 = (long long)tile * 128 + wq * 32;
                            psg_store_rm32(v, stage_rm + warp * 256, lane, op.rm + row0 * op.rm_stride + c0l + c, op.rm_stride,
                                           [&](int i) { return row0 + i < a.rows; });
                        }
                        if (op.mglobal) op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r] = w;
                    }
                    if (c < nl) {
                        float v[16];
                        tc::tmem_ld16(tl + (uint32_t)c, v);
                        unsigned w = 0;
                        if (op.relu) w = psg_relu_bias_bits<16>(v, sbias + op.boff + c0l + c);
                        if (valid) {
                            if (!op.rm_only) {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    tv_st(op.out, row, ((c0l + c) >> 2) + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
                            }
                            if (op.rm) {
                                float4 *d = reinterpret_cast<float4 *>(op.rm + row * op.rm_stride + c0l + c);
#pragma unroll
                                for (int j = 0; j < 4; ++j) d[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                            }
                        }
                        if (op.mglobal) op.mglobal[((size_t)tile * words + w0l + (c >> 5)) * 128 + r] = w;
                    }
                } else if (op.epi == EPI_MAXPOOL) {
                    // neighbourhood max through a shared-memory transpose (psg_epi.cuh); the per-tile mask area
                    // is unused by forward set-abstraction programs and serves as the warps' scratch.
                    // (Everything here stays in registers: with the shared-memory carve-out at its maximum
                    // there is next to no L1, so a local-memory array costs an L2 round trip per access.)
                    float *scratch = reinterpret_cast<float *>(mbits) + wq * 1024;
                    const long long g0 = ((long long)tile * 128 + wq * 32) / K;
                    const float *bs = sbias + op.boff + c0l;
                    auto emit1 = [&](long long gg, int col, float best, int arg) {
                        if (gg * K < a.rows) {
                            op.out.base[tv_off(op.out, gg, (c0l + col) >> 2) + ((c0l + col) & 3)] = best;
                            op.arg[gg * op.argC + op.arg0 + c0l + col] = (unsigned char)arg;
                        }
                    };
                    for (int c = 0; c < nl; c += 32) {
                        float v[32];
                        const bool full = c + 32 <= nl;                 // else a 16-column tail
                        if (full) tc::tmem_ld32(tl + (uint32_t)c, v);
                        else {
                            tc::tmem_ld16(tl + (uint32_t)c, v);
#pragma unroll
                            for (int i = 16; i < 32; ++i) v[i] = 0.f;
                        }
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 b = (full || q < 4) ? *reinterpret_cast<const float4 *>(bs + c + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                            v[4 * q] = fmaxf(v[4 * q] + b.x, 0.f); v[4 * q + 1] = fmaxf(v[4 * q + 1] + b.y, 0.f);
                            v[4 * q + 2] = fmaxf(v[4 * q + 2] + b.z, 0.f); v[4 * q + 3] = fmaxf(v[4 * q + 3] + b.w, 0.f);
                        }
                        const bool mine = full || lane < 16;
                        if (K == 32) {
                            float best[1]; int arg[1];
                            psg_pool_transposed<32, 32>(v, scratch, lane, best, arg);
                            if (mine) emit1(g0, c + lane, best[0], arg[0]);
                        } else {
                            float best[2]; int arg[2];
                            psg_pool_transposed<16, 32>(v, scratch, lane, best, arg);
                            if (mine) { emit1(g0, c + lane, best[0], arg[0]); emit1(g0 + 1, c + lane, best[1], arg[1]); }
                        }
                    }
                } else if (op.epi == EPI_HEAD) {          // CS == 1 only (16 logit columns do not split)
                    float v[16], dz[16];
                    tc::tmem_ld16(tl, v);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] += sbias[op.boff + i];
                    if (!a.backward) {
                        if (valid) {
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                tv_st(a.zout, row, c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
                        }
                    } else {
                        const long long rr = valid ? row : 0;
                        if (a.loss_kind == 0) {
                            psg_dz_generic(v, a.ncls, a.dlogp + rr * a.ncls, dz);
                        } else if (a.loss_kind == 1) {
                            psg_dz_ce_row(v, a.ncls, a.target >= 0 ? a.target : a.labels[rr], a.scale, dz);
                        } else {
                            int h;
                            const float f = psg_dz_cw_row(v, a.ncls, a.target >= 0 ? a.target : a.labels[rr], a.kappa, a.scale, dz, h);
                            if (valid && a.loss_rows) a.loss_rows[row] = f;
                            if (valid && a.hit) a.hit[row] = (unsigned char)h;
                        }
                        if (!valid) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) dz[i] = 0.f;
                        }
                        put16(0, dz);
                    }
                }
                // EPI_NONE: the accumulator is continued by the next op
                if (tr && tn < 510) tr[tn++] = clock64();
            }
            tc::fence_before_sync();
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (CS > 1) tc::cluster_sync_all();            // no CTA exits while a peer may still write into it
    if (warp == NG * 4) tc::tmem_dealloc(tmem, ncols);
}

int g_sms = 0;
long long *g_trace = nullptr;
int g_trace_cap = 0, g_trace_n = 0;
constexpr size_t kSmemMax = 232448 - 256;      // 227 KB per CTA minus the static barriers

inline uint32_t pow2cols(int n) { uint32_t c = 32; while ((int)c < n) c <<= 1; return c; }

struct Builder {
    TileArgs a;
    int amax_cols = 0;    // widest A operand (columns)
    int nmax = 0;         // widest accumulator
    bool ok = true;
    bool x3 = false;      // 3xTF32 program: every op carries wlo, the operand holds [A | A_lo]
    Builder() { memset(&a, 0, sizeof(a)); }
    TileOp *add(const float *w, int wstride, int wrow0, int wplane0, int n, int planes, int aplane0)
    {
        if (a.nops >= kMaxOps || n % 16 || n < 16 || n > 256 || planes % 2 || planes < 2) { ok = false; return &a.ops[0]; }
        TileOp &o = a.ops[a.nops++];
        memset(&o, 0, sizeof(o));
        o.w = w; o.wstride = wstride; o.wrow0 = wrow0; o.wplane0 = wplane0; o.n = n; o.planes = planes; o.aplane0 = aplane0;
        o.slot = -1;
        if ((aplane0 + planes) * 4 > amax_cols) amax_cols = (aplane0 + planes) * 4;
        if (n > nmax) nmax = n;
        return &o;
    }
    void want_a(int cols) { if (cols > amax_cols) amax_cols = cols; }
};

// cluster size for a program: the largest CS in {4, 2} such that every tile still gets its own cluster
// in one wave and every op's columns split into whole 16-column (32 for masked layers) slices
int pick_cluster(const TileArgs &a, int ntiles, int sms)
{
    for (int cs = 4; cs >= 2; cs >>= 1) {
        if (ntiles * cs > sms) continue;
        bool ok = true;
        for (int o = 0; o < a.nops && ok; ++o) {
            const TileOp &op = a.ops[o];
            if (op.epi == EPI_HEAD) ok = false;
            const int unit = (op.epi == EPI_RELU || op.epi == EPI_MASK || op.mglobal) ? 32 : 16;
            if (op.n % (unit * cs)) ok = false;
        }
        if (ok) return cs;
    }
    return 1;
}

template <int NG, int CS, bool TS = false, bool X3 = false>
int launch_tile(const TileArgs &a, int grid, size_t smem, cudaStream_t st)
{
    static PsgDeviceOnce attr_once;
    if (attr_once.need()) {
        if (cudaFuncSetAttribute(tile_kernel<NG, CS, TS, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax) != cudaSuccess)
            return PSG_ECUDA;
        attr_once.mark();
    }
    if (psg_launch_pdl(tile_kernel<NG, CS, TS, X3>, dim3((unsigned)grid), dim3(NG * 128 + 64), smem, st, CS, a) != cudaSuccess)
        return PSG_ECUDA;
    return PSG_OK;
}

// A-operand-in-tensor-memory mode: row-local chains whose only refill is the interpolation (fp1 + head).  The operand
// region needs whole 32-column stores and, with the accumulator, has to fit the 512 TMEM columns NG times.
bool ts_eligible(const Builder &b, int ng)
{
    const TileArgs &a = b.a;
    if (b.amax_cols % 32) return false;
    for (int o = 0; o < a.nops; ++o) {
        const TileOp &op = a.ops[o];
        if (op.pre != PRE_NONE && op.pre != PRE_FP) return false;
        if (op.pre == PRE_FP && (a.src.lcols != 0 || a.src.icols % 32)) return false;
        if (op.epi == EPI_MAXPOOL) return false;
        if ((op.epi == EPI_RELU || op.epi == EPI_MASK) && op.n % 16) return false;
    }
    return (int)pow2cols(ng * ((int)pow2cols(b.nmax) + b.amax_cols)) <= 512;
}

// choose cluster size / NG / stage size to fit shared memory, fill the derived fields, launch
int launch_program(Builder &b, long long rows, cudaStream_t st)
{
    if (!b.ok || b.a.nops < 1) return PSG_EUNSUPPORTED;
    TileArgs &a = b.a;
    if (g_sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            return PSG_ECUDA;
    }
    a.rows = rows; a.ntiles = (int)((rows + 127) / 128);
    a.trace = psg_tile_trace_slot();
    a.abytes = b.amax_cols * 512;
    const int cs = pick_cluster(a, a.ntiles, g_sms);
    a.tcols = (int)pow2cols(b.nmax / cs);
    a.bias_floats = 0;
    for (int o = 0; o < a.nops; ++o) {
        a.ops[o].boff = a.bias_floats;
        if (a.ops[o].bias) a.bias_floats += (a.ops[o].n + 3) & ~3;
    }
    // per-tile mask area: (highest slot + 1) x (words of the widest masked layer) x 128 rows
    int nslots = 0;
    a.mwords = 0;
    for (int o = 0; o < a.nops; ++o) {
        if (a.ops[o].slot < 0) continue;
        if (a.ops[o].slot + 1 > nslots) nslots = a.ops[o].slot + 1;
        if ((a.ops[o].n + 31) / 32 > a.mwords) a.mwords = (a.ops[o].n + 31) / 32;
    }
    a.mbytes = nslots * a.mwords * 128 * 4;
    for (int o = 0; o < a.nops; ++o)
        if (a.ops[o].epi == EPI_MAXPOOL && a.mbytes < 16384) a.mbytes = 16384;     // pool scratch: 4 KB per worker warp
    bool scatters = false, mirrors = false;
    for (int o = 0; o < a.nops; ++o) {
        scatters = scatters || a.ops[o].pre == PRE_SCATTER;
        mirrors = mirrors || (a.ops[o].epi == EPI_STORE && a.ops[o].rm);
    }
    a.rmstage = 0;
    auto need = [&](int ng, int stg) {
        return (size_t)ng * a.abytes + (size_t)kStages * stg + (size_t)ng * a.mbytes + (size_t)a.bias_floats * 4 +
               ((scatters || a.rmstage) ? (size_t)ng * 4 * 32 * 20 : 0) + (a.rmstage ? (size_t)ng * 4 * 4096 : 0) + 128;
    };
    // two tiles in flight share every weight stage; with few tiles one tile per CTA spreads them over more SMs
    int ng = (cs == 1 && a.ntiles > g_sms && a.tcols * 2 <= 512 && need(2, 16 * 1024) <= kSmemMax) ? 2 : 1;
    if (b.x3) {
        // operand = [A | A_lo]: the residual copy starts at the widest operand's width, one tile in flight, tensor memory only
        if (cs != 1) return PSG_EUNSUPPORTED;
        ng = 1;
        a.lo_off = (b.amax_cols + 31) / 32 * 32;
        b.amax_cols = 2 * a.lo_off;
    }
    const bool ts = cs == 1 && ts_eligible(b, ng);
    if (b.x3 && !ts) return PSG_EUNSUPPORTED;
    if (ts) { a.abytes = 0; a.acols = b.amax_cols; }          // no operand buffer in shared memory: room for 64 KB stages
    int stage = (ts && need(ng, 64 * 1024) <= kSmemMax) ? 64 * 1024 : need(ng, 32 * 1024) <= kSmemMax ? 32 * 1024 : 16 * 1024;
    if (need(ng, stage) > kSmemMax || a.tcols * ng > 512) return PSG_EUNSUPPORTED;
    if (mirrors) {                   // staging for coalesced row-major stores, if it fits without shrinking the weight stages
        a.rmstage = 1;
        if (need(ng, stage) > kSmemMax) a.rmstage = 0;
    }
    a.stage_bytes = stage;
    for (int o = 0; o < a.nops; ++o) {
        TileOp &op = a.ops[o];
        int pps = stage / ((op.n / cs) * 16);
        pps &= ~1;
        if (pps < 2) return PSG_EUNSUPPORTED;
        op.pps = pps < op.planes ? pps : op.planes;
    }
    const size_t smem = need(ng, stage);
    int rc;
    if (cs == 1) {
        const int want = (a.ntiles + ng - 1) / ng;
        const int grid = want < g_sms ? want : g_sms;
        if (b.x3) rc = launch_tile<1, 1, true, true>(a, grid, smem, st);
        else if (ts) rc = ng == 2 ? launch_tile<2, 1, true>(a, grid, smem, st) : launch_tile<1, 1, true>(a, grid, smem, st);
        else rc = ng == 2 ? launch_tile<2, 1>(a, grid, smem, st) : launch_tile<1, 1>(a, grid, smem, st);
    } else {
        const int grid = a.ntiles * cs;                     // one cluster per tile, all resident in one wave
        rc = cs == 4 ? launch_tile<1, 4>(a, grid, smem, st) : launch_tile<1, 2>(a, grid, smem, st);
    }
    if (rc != PSG_OK) return rc;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

}  // namespace

// -------------------------------------------------------------------------------------------------
// fp1 + head (forward [+ loss + backward])
// -------------------------------------------------------------------------------------------------
int psg_chain_fused(const PsgChain &c, cudaStream_t st)
{
    if (c.nlayers < 1 || c.nlayers > kMaskSlots || c.kin % 16 || c.kin > 256 || c.ncls > kPsgMaxCls) return PSG_EUNSUPPORTED;
    Builder b;
    b.x3 = c.head_wf_lo != nullptr;
    int kprev = c.kin;
    for (int j = 0; j < c.nlayers; ++j) {          // hidden layers: bias + ReLU, bits kept in shared-memory slot j
        if (c.n[j] > 256) return PSG_EUNSUPPORTED;
        TileOp *o = b.add(c.wf[j], c.nwf[j], 0, 0, c.n[j], kprev / 4, 0);
        o->wlo = b.x3 ? c.wf_lo[j] : nullptr;
        o->epi = EPI_RELU; o->bias = c.bias[j]; o->slot = j;
        if (j == 0) o->pre = PRE_FP;
        kprev = c.n[j];
    }
    {                                               // head: N = 16 logits columns (zero-padded classes)
        TileOp *o = b.add(c.head_wf, c.head_nwf, 0, 0, 16, kprev / 4, 0);
        o->wlo = c.head_wf_lo;
        o->epi = EPI_HEAD; o->bias = c.head_bias;
    }
    if (c.backward) {
        {                                           // d hidden_last = dz W_head, masked by the last hidden layer's bits
            TileOp *o = b.add(c.head_wb, c.head_nwb, 0, 0, kprev, 16 / 4, 0);
            o->wlo = c.head_wb_lo;
            o->epi = EPI_MASK; o->slot = c.nlayers - 1;
        }
        for (int j = c.nlayers - 1; j >= 0; --j) {
            const int nin = j > 0 ? c.n[j - 1] : c.kin;
            TileOp *o = b.add(c.wb[j], c.nwb[j], 0, 0, nin, c.n[j] / 4, 0);
            o->wlo = b.x3 ? c.wb_lo[j] : nullptr;
            if (j > 0) { o->epi = EPI_MASK; o->slot = j - 1; }
            else { o->epi = EPI_STORE; o->out = c.dI; o->rm = c.dI_rm; o->rm_stride = c.kin; o->rm_only = (c.dI_rm && c.rm_only) ? 1 : 0; }
        }
    }
    TileArgs &a = b.a;
    a.src.isrc = c.src; a.src.iS = c.S; a.src.iNf = c.Nf; a.src.icols = c.kin; a.src.iplane0 = 0;
    a.src.nn_idx = c.nn_idx; a.src.nn_w = c.nn_w; a.src.lcols = 0;
    a.src.irm = c.src_rm; a.src.irm_stride = c.kin;
    a.backward = c.backward; a.ncls = c.ncls; a.loss_kind = c.loss_kind; a.target = c.target; a.labels = c.labels;
    a.scale = c.scale; a.kappa = c.kappa; a.dlogp = c.dlogp; a.loss_rows = c.loss_rows; a.hit = c.hit;
    a.zout = c.zout;
    return launch_program(b, c.rows, st);
}

// -------------------------------------------------------------------------------------------------
// wide set-abstraction level (weights streamed)
// -------------------------------------------------------------------------------------------------
bool psg_sa_streamable(int K, int gpad, int n0, int n1, int n2)
{
    if (K != 16 && K != 32) return false;
    if (gpad % 16 || n0 % 16 || n1 % 16 || n2 % 16) return false;
    if (gpad > 288 || n0 > 256 || n1 > 256 || n2 > 512) return false;
    return true;
}

int psg_sa_stream_fwd(const PsgSaFused &f, cudaStream_t st)
{
    Builder b;
    TileOp *o = b.add(f.wf[0], f.nwf[0], 0, 0, f.n[0], f.gpad / 4, 0);
    o->pre = PRE_GROUP; o->epi = EPI_RELU; o->bias = f.bias[0]; o->mglobal = f.m0;
    o = b.add(f.wf[1], f.nwf[1], 0, 0, f.n[1], f.n[0] / 4, 0);
    o->epi = EPI_RELU; o->bias = f.bias[1]; o->mglobal = f.m1;
    for (int c0 = 0; c0 < f.n[2]; c0 += 256) {
        const int n = f.n[2] - c0 < 256 ? f.n[2] - c0 : 256;
        o = b.add(f.wf[2], f.nwf[2], c0, 0, n, f.n[1] / 4, 0);
        o->epi = EPI_MAXPOOL; o->bias = f.bias[2] + c0;
        o->out = f.out; o->out.c0 += c0 / 4;
        o->arg = f.arg; o->argC = f.n[2]; o->arg0 = c0;
    }
    TileSrc &s = b.a.src;
    s.feats = f.feats; s.D = f.D; s.gpad = f.gpad; s.xyz = f.xyz; s.cloud_stride = f.cloud_stride; s.nclouds = f.nclouds;
    s.Nsrc = f.Nsrc; s.new_xyz = f.new_xyz; s.idx = f.idx; s.S = f.S; s.K = f.K;
    return launch_program(b, f.rows, st);
}

int psg_sa_stream_bwd(const PsgSaFused &f, TView dout, TView dG, int gcols, float *dG_rm, int rm_only, cudaStream_t st)
{
    Builder b;
    TileOp *o = nullptr;
    // dY1 = dY2 W2, contraction over n2 in slabs (the scatter refills the A buffer per slab); a slab is no
    // wider than the hidden layers need the buffer to be anyway, so narrow levels keep two tiles in flight
    int slab = f.n[0] > f.n[1] ? f.n[0] : f.n[1];
    slab = slab < 128 ? 128 : (slab > 256 ? 256 : slab);
    for (int c0 = 0; c0 < f.n[2]; c0 += slab) {
        const int kc = f.n[2] - c0 < slab ? f.n[2] - c0 : slab;
        o = b.add(f.wb[2], f.nwb[2], 0, c0 / 4, f.n[1], kc / 4, 0);
        o->pre = PRE_SCATTER; o->pre_a = c0; o->accumulate = c0 > 0 ? 1 : 0; o->epi = EPI_NONE;
    }
    o->epi = EPI_MASK; o->mglobal = f.m1;
    o = b.add(f.wb[1], f.nwb[1], 0, 0, f.n[0], f.n[1] / 4, 0);
    o->epi = EPI_MASK; o->mglobal = f.m0;
    for (int c0 = 0; c0 < gcols; c0 += 256) {
        const int n = gcols - c0 < 256 ? gcols - c0 : 256;
        o = b.add(f.wb[0], f.nwb[0], c0, 0, n, f.n[0] / 4, 0);
        o->epi = EPI_STORE; o->out = dG; o->out.c0 += c0 / 4;
        if (dG_rm) { o->rm = dG_rm + c0; o->rm_stride = f.gpad; o->rm_only = rm_only; }
    }
    TileSrc &s = b.a.src;
    s.K = f.K; s.dout = dout; s.outv = f.out; s.sarg = f.arg; s.sargC = f.n[2];
    return launch_program(b, f.rows, st);
}

// -------------------------------------------------------------------------------------------------
// feature-propagation level (weights streamed)
// -------------------------------------------------------------------------------------------------
// does the whole concatenated input of level f fit the operand buffer next to two 16 KB weight stages?
static bool fp_fits_whole(const PsgFpStream &f)
{
    size_t bias = 0;
    for (int j = 0; j < f.nl; ++j) bias += (size_t)f.n[j] * 4;
    return (size_t)(f.C1 + f.C2) * 512 + 2 * 16 * 1024 + bias + 128 <= kSmemMax;
}

bool psg_fp_streamable(const PsgFpStream &f, bool forward)
{
    if (f.nl < 1 || f.nl > 3 || f.C1 % 16 || f.C2 % 16) return false;
    for (int j = 0; j < f.nl; ++j)
        if (f.n[j] % 32 || f.n[j] > 256) return false;
    // Forward inputs wider than the operand buffer run per layer: for the levels that have them (FP4: 1024 rows x 768
    // columns at B = 16) the per-layer GEMMs with their deep operand ring and 64 column-split CTAs measured faster than
    // a tile program contracting the input in 256-column slabs (fp4 forward 45 us vs 95 us).
    return !forward || fp_fits_whole(f);
}

// [skip | interp] -> nl x (conv + folded BN + ReLU); last layer stored (it is the next level's
// interpolation source and its ReLU mask), hidden layers leave their ReLU bits in `m[j]`
int psg_fp_stream_fwd(const PsgFpStream &f, cudaStream_t st)
{
    Builder b;
    int kprev = f.C1 + f.C2;
    for (int j = 0; j < f.nl; ++j) {
        TileOp *o = b.add(f.wf[j], f.nwf[j], 0, 0, f.n[j], kprev / 4, 0);
        if (j == 0) { o->pre = PRE_FP; o->pre_a = 0; }
        o->bias = f.bias[j];
        if (j + 1 < f.nl) { o->epi = EPI_RELU; o->mglobal = f.m[j]; }
        else { o->epi = EPI_STORE; o->relu = 1; o->out = f.y_last; o->rm = f.y_last_rm; o->rm_stride = f.n[j]; }
        kprev = f.n[j];
    }
    TileSrc &s = b.a.src;
    s.lsrc = f.skip; s.lcols = f.C1;
    s.isrc = f.coarse; s.iS = f.S; s.iNf = f.Nf; s.icols = f.C2; s.iplane0 = f.C1 / 4; s.nn_idx = f.nn_idx; s.nn_w = f.nn_w;
    s.irm = f.coarse_rm; s.irm_stride = f.C2;
    return launch_program(b, f.rows, st);
}

// the store epilogue writes its second destination in whole 32-column groups, and only the first op (columns 0..255)
// carries it
int psg_fp_stream_skip_cols(const PsgFpStream &f)
{
    if (f.C1 % 32) return 0;
    return f.C1 < 256 ? f.C1 : 256;
}

// dY_last (pre-activation gradient, already masked) -> dgrad chain -> d[skip | interp] stored to dcat
int psg_fp_stream_bwd(const PsgFpStream &f, TView dy_last, TView dcat, float *dcat_rm, TView dskip, cudaStream_t st)
{
    Builder b;
    const int skip_cols = dskip.base ? psg_fp_stream_skip_cols(f) : 0;
    for (int j = f.nl - 1; j >= 0; --j) {
        const int nin = j > 0 ? f.n[j - 1] : f.C1 + f.C2;
        if (j > 0) {
            TileOp *o = b.add(f.wb[j], f.nwb[j], 0, 0, nin, f.n[j] / 4, 0);
            o->epi = EPI_MASK; o->mglobal = f.m[j - 1];
            if (j == f.nl - 1) o->pre = PRE_LOAD;
        } else {
            for (int c0 = 0; c0 < nin; c0 += 256) {
                const int n = nin - c0 < 256 ? nin - c0 : 256;
                TileOp *o = b.add(f.wb[0], f.nwb[0], c0, 0, n, f.n[0] / 4, 0);
                o->epi = EPI_STORE; o->out = dcat; o->out.c0 += c0 / 4;
                if (dcat_rm) { o->rm = dcat_rm + c0; o->rm_stride = f.C1 + f.C2; }
                if (c0 == 0 && skip_cols) { o->out2 = dskip; o->out2_cols = skip_cols; }
                if (f.nl == 1 && c0 == 0) o->pre = PRE_LOAD;
            }
        }
    }
    TileSrc &s = b.a.src;
    s.lsrc = dy_last; s.lcols = f.n[f.nl - 1];
    b.want_a(f.n[f.nl - 1]);
    return launch_program(b, f.rows, st);
}

long long *psg_tile_trace_slot() { return (g_trace && g_trace_n < g_trace_cap) ? g_trace + (size_t)(g_trace_n++) * 2048 : nullptr; }
void psg_tile_set_trace(long long *buf, int nlaunches) { g_trace = buf; g_trace_cap = nlaunches; g_trace_n = 0; }
