// gemm_tc.cu -- tcgen05 / TMEM TF32 GEMM for the shared 1x1-conv MLPs (same interface and operand
// layout as gemm_simt.cu):   Out[M, Nout] = epilogue( [A1 | A2][M, K] * W[Nout, K]^T )
//
// One CTA computes a 128 x BN output tile (BN <= 128).  Warp 0 (one lane) streams the operands
// with 1-D bulk async copies: a 128-row activation tile of T-layout is a run of whole 2 KB chunk
// planes, i.e. already the K-major no-swizzle UMMA canonical layout, and the packed weights
// [K/4][Nw][4] are the same layout for the B operand.  Warp 1 allocates TMEM and (one lane) issues
// tcgen05.mma.kind::tf32 (M = 128, N = BN, K = 8 per instruction) into a TMEM accumulator, handing
// shared-memory stages back through tcgen05.commit -> mbarrier.  Warps 2-5 read the accumulator
// with tcgen05.ld (thread = row), apply bias / ReLU / ReLU-mask and write T-layout rows as
// coalesced 16-byte pieces.
#include <cstring>
#include "psg_common.cuh"
#include "psg_internal.h"
#include "psg_tc.cuh"
#include "psg_tmap.cuh"

namespace {

constexpr int kMaxStages = 12;
// chunk planes (4 floats of K each) per stage: 16 (32 KB of activations) -- the producer's per-stage bookkeeping (wait,
// expect_tx, issue: ~350 ns, tools/l2_stream_bench.py) bounds the K loop, not the L2 (>= 100 GB/s per SM), so stages are
// as large as the ring allows; the 3xTF32 kernel keeps 8 (its stages hold A, A_lo, W_hi and W_lo)
constexpr int kBNMax = 128;
constexpr int kThreads = 192;
constexpr int kRingBytes = 200 * 1024;        // operand ring: as many stages as fit (the K loop is a latency chain)
constexpr int kSmemBytes = kRingBytes + 1024;

__device__ __forceinline__ long long gtimer()
{
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// X3: error-compensated TF32 ("3xTF32"), fp32-grade products on the tensor cores.  tcgen05.mma.kind::tf32 reads the top
// 19 bits of each fp32 operand, so A as it lies in shared memory IS A_hi; the four epilogue warps, idle during the K
// loop, write A_lo = A - A_hi (exact in fp32) next to every stage as it lands; the weights arrive pre-split from the host
// (W_hi = nearest TF32 of W, W_lo = nearest TF32 of W - W_hi).  Three MMAs per K step accumulate A_lo W_hi + A_hi W_lo +
// A_hi W_hi into the same TMEM accumulator; the dropped A_lo W_lo term is 2^-22 relative.
template <int EPI, bool X3, int KB>
__global__ void __launch_bounds__(kThreads) gemm_tc_kernel(PsgGemmArgs g, int bn_tile, int kStages, long long *trace,
                                                           const __grid_constant__ CUtensorMap wmap, int use_map)
{
    constexpr int kBlk = KB;
    constexpr int kABytes = kBlk * 2048;
    long long *tr = (trace && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 64) ? trace : nullptr;   // first epilogue thread
    if (tr) tr[0] = gtimer();
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar_full[kMaxStages], bar_empty[kMaxStages], bar_split[kMaxStages], bar_acc;
    __shared__ uint32_t tmem_slot;

    // 1024-byte aligned operand staging area: [A stages][A_lo stages (X3)][B stages (X3: hi | lo per stage)]
    const uint32_t sbase = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int kBHalf = kBlk * bn_tile * 16;
    const int kBBytes = X3 ? 2 * kBHalf : kBHalf;
    const uint32_t sA = sbase, sAlo = sbase + kStages * kABytes, sB = sbase + (X3 ? 2 : 1) * kStages * kABytes;
    unsigned char *pA = smem_raw + (sbase - tc::smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row0 = (long long)blockIdx.x * 128;
    const int n0 = blockIdx.y * bn_tile;
    const int BN = min(bn_tile, g.nout_pad - n0);
    const uint32_t ncols = tc::next_pow2_cols(BN);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            tc::mbar_init(tc::smem_u32(&bar_full[s]), 1); tc::mbar_init(tc::smem_u32(&bar_empty[s]), 1);
            tc::mbar_init(tc::smem_u32(&bar_split[s]), 128);
        }
        tc::mbar_init(tc::smem_u32(&bar_acc), 1);
        tc::fence_mbar_init();
    }
    if (warp == 1) tc::tmem_alloc(tc::smem_u32(&tmem_slot), ncols);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tr) tr[1] = gtimer();
    tc::pdl_launch_dependents();
    if (warp != 0) tc::pdl_wait();   // launched with programmatic stream serialization: the prologue overlapped the predecessor
    if (tr) tr[2] = gtimer();        // (the producer warp waits after it has requested the first weight stages)
    const uint32_t tmem = tmem_slot;

    if (warp == 0) {
        // ---- producer: the whole warp issues a stage's copies (lane 0: barrier bookkeeping + the A tile, lane j:
        // weight plane j, or lane 1 one tiled TMA copy).  One thread issuing the nine copies of a stage back to back
        // cost ~80 ns per copy.  The weights of the first ring-full of stages are requested BEFORE
        // griddepcontrol.wait (they are constants), the activations after it. ----
        const int s0n = (g.k1chunks + kBlk - 1) / kBlk, s1n = (g.k2chunks + kBlk - 1) / kBlk, total = s0n + s1n;
        auto stage_of = [&](int it, int &srcI, int &c, int &kglob, int &n) {
            srcI = it < s0n ? 0 : 1;
            c = (srcI == 0 ? it : it - s0n) * kBlk;
            kglob = srcI == 0 ? 0 : g.k1chunks;
            n = min(kBlk, (srcI == 0 ? g.k1chunks : g.k2chunks) - c);
        };
        auto issue_w = [&](int s, int c, int kglob, int n, uint32_t full) {
            if (X3) {
                // lanes 1..n: the hi plane, lanes 9..8+n: the lo plane of the same K chunk
                const int j = (lane - 1) % kBlk;
                if (lane >= 1 && lane <= 2 * kBlk && j < n) {
                    const float *w = lane <= kBlk ? g.W : g.Wlo;
                    tc::bulk_g2s(sB + s * kBBytes + (lane <= kBlk ? 0 : kBHalf) + j * BN * 16, w + ((size_t)(kglob + c + j) * g.Nw + n0) * 4,
                                 (uint32_t)(BN * 16), full);
                }
            } else if (use_map && BN == bn_tile && n == kBlk) {
                // the box is always kBlk planes: a short stage (a source whose width is not a whole number of stages,
                // e.g. 20 + 12 planes) would deliver more bytes than its expect_tx and never complete; it takes the
                // per-plane copies below
                if (lane == 1) psg_tmap_load(sB + s * kBBytes, &wmap, n0, kglob + c, full);
            } else if (lane >= 1 && lane <= n) {
                const int j = lane - 1;
                tc::bulk_g2s(sB + s * kBBytes + j * BN * 16, g.W + ((size_t)(kglob + c + j) * g.Nw + n0) * 4, (uint32_t)(BN * 16), full);
            }
        };
        const int pre = min(total, kStages);
        for (int it = 0; it < pre; ++it) {
            int srcI, c, kglob, n;
            stage_of(it, srcI, c, kglob, n);
            const uint32_t full = tc::smem_u32(&bar_full[it]);
            if (lane == 0) tc::mbar_expect_tx(full, (uint32_t)(n * 2048 + (X3 ? 2 : 1) * n * BN * 16));
            __syncwarp();
            issue_w(it, c, kglob, n, full);
        }
        tc::pdl_wait();
        if (lane == 0) {
            for (int it = 0; it < pre; ++it) {
                int srcI, c, kglob, n;
                stage_of(it, srcI, c, kglob, n);
                const TView &src = srcI == 0 ? g.A1 : g.A2;
                tc::bulk_g2s(sA + it * kABytes, src.base + tv_off(src, row0, c), (uint32_t)(n * 2048), tc::smem_u32(&bar_full[it]));
            }
        }
        for (int it = pre; it < total; ++it) {
            int srcI, c, kglob, n;
            stage_of(it, srcI, c, kglob, n);
            const TView &src = srcI == 0 ? g.A1 : g.A2;
            const int s = it % kStages;
            const uint32_t ph = (uint32_t)(it / kStages) & 1u;
            const uint32_t full = tc::smem_u32(&bar_full[s]);
            if (lane == 0) {
                tc::mbar_spin(tc::smem_u32(&bar_empty[s]), ph ^ 1u);
                tc::mbar_expect_tx(full, (uint32_t)(n * 2048 + (X3 ? 2 : 1) * n * BN * 16));
            }
            __syncwarp();
            if (lane == 0) tc::bulk_g2s(sA + s * kABytes, src.base + tv_off(src, row0, c), (uint32_t)(n * 2048), full);
            issue_w(s, c, kglob, n, full);
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer ----
            const uint32_t idesc = tc::idesc_tf32(128, BN);
            int it = 0;
            uint32_t acc = 0;
            for (int srcI = 0; srcI < 2; ++srcI) {
                const int kch = srcI == 0 ? g.k1chunks : g.k2chunks;
                for (int c = 0; c < kch; c += kBlk, ++it) {
                    const int n = min(kBlk, kch - c);
                    const int s = it % kStages;
                    const uint32_t ph = (uint32_t)(it / kStages) & 1u;
                    tc::mbar_wait(tc::smem_u32(X3 ? &bar_split[s] : &bar_full[s]), ph);
                    tc::fence_after_sync();
                    for (int j = 0; j < n; j += 2) {
                        const uint64_t ad = tc::smem_desc(sA + s * kABytes + j * 2048, 2048, 128);
                        const uint64_t bd = tc::smem_desc(sB + s * kBBytes + j * BN * 16, (uint32_t)(BN * 16), 128);
                        if (X3) {
                            const uint64_t al = tc::smem_desc(sAlo + s * kABytes + j * 2048, 2048, 128);
                            const uint64_t bl = tc::smem_desc(sB + s * kBBytes + kBHalf + j * BN * 16, (uint32_t)(BN * 16), 128);
                            tc::mma_tf32(tmem, al, bd, idesc, acc);       // small terms first
                            tc::mma_tf32(tmem, ad, bl, idesc, 1u);
                            tc::mma_tf32(tmem, ad, bd, idesc, 1u);
                        } else
                        tc::mma_tf32(tmem, ad, bd, idesc, acc);
                        acc = 1;
                    }
                    tc::mma_commit(tc::smem_u32(&bar_empty[s]));
                }
            }
            tc::mma_commit(tc::smem_u32(&bar_acc));
        }
    } else {
        // ---- epilogue: warp q owns TMEM lanes [32q, 32q + 32) ----
        const int q = warp & 3;
        const long long row = row0 + q * 32 + lane;
        if (X3) {
            // A_lo of every stage as it lands (the K loop's stage order; these warps have nothing else to do until the
            // accumulator is complete)
            const int tid = threadIdx.x - 64;
            int it = 0;
            for (int srcI = 0; srcI < 2; ++srcI) {
                const int kch = srcI == 0 ? g.k1chunks : g.k2chunks;
                for (int c = 0; c < kch; c += kBlk, ++it) {
                    const int n = min(kBlk, kch - c);
                    const int s = it % kStages;
                    const uint32_t ph = (uint32_t)(it / kStages) & 1u;
                    tc::mbar_wait(tc::smem_u32(&bar_full[s]), ph);
                    const float4 *src = reinterpret_cast<const float4 *>(pA + (size_t)s * kABytes);
                    float4 *dst = reinterpret_cast<float4 *>(pA + (size_t)(kStages + s) * kABytes);
#pragma unroll 4
                    for (int i = tid; i < n * 128; i += 128) {
                        const float4 a = src[i];
                        float4 l;
                        l.x = a.x - __uint_as_float(__float_as_uint(a.x) & 0xFFFFE000u);
                        l.y = a.y - __uint_as_float(__float_as_uint(a.y) & 0xFFFFE000u);
                        l.z = a.z - __uint_as_float(__float_as_uint(a.z) & 0xFFFFE000u);
                        l.w = a.w - __uint_as_float(__float_as_uint(a.w) & 0xFFFFE000u);
                        dst[i] = l;
                    }
                    tc::fence_async_smem();
                    tc::mbar_arrive(tc::smem_u32(&bar_split[s]));
                }
            }
        }
        tc::mbar_wait(tc::smem_u32(&bar_acc), 0);
        tc::fence_after_sync();
        if (tr) tr[3] = gtimer();
        for (int c16 = 0; c16 < BN; c16 += 16) {
            float v[16];
            tc::tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c16, v);
            const int col = n0 + c16;
            if (EPI == PSG_EPI_BIAS_RELU || EPI == PSG_EPI_BIAS) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    v[i] += __ldg(g.bias + col + i);
                    if (EPI == PSG_EPI_BIAS_RELU) v[i] = fmaxf(v[i], 0.f);
                }
            }
            if (EPI == PSG_EPI_MASK) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 y = tv_ld(g.Mask, row, (col >> 2) + c);
                    v[4 * c + 0] = y.x > 0.f ? v[4 * c + 0] : 0.f;
                    v[4 * c + 1] = y.y > 0.f ? v[4 * c + 1] : 0.f;
                    v[4 * c + 2] = y.z > 0.f ? v[4 * c + 2] : 0.f;
                    v[4 * c + 3] = y.w > 0.f ? v[4 * c + 3] : 0.f;
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                tv_st(g.Out, row, (col >> 2) + c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
            if (g.Out2.base && col + 16 <= g.out2_cols) {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    tv_st(g.Out2, row, (col >> 2) + c, make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
            }
        }
    }
    if (tr) tr[4] = gtimer();
    tc::fence_before_sync();
    __syncthreads();
    if (tr) { tr[5] = gtimer(); tr[6] = g.mtiles; tr[7] = (long long)(g.k1chunks + g.k2chunks) * 4; tr[8] = g.nout_pad; tr[9] = bn_tile; }
    if (warp == 1) tc::tmem_dealloc(tmem, ncols);
}

// ring depth of the many-tile layers, and what "many" means: two CTAs per SM instead of one behind the full ring
// (measured: MSG B = 64 275 -> 295 steps/s, 3xTF32 mode 409 -> 536)
constexpr int kNstPlain = 2, kNstX3 = 1, kBigCtas = 148;

template <int EPI, bool X3, int KB>
int launch_kb(const PsgGemmArgs &g, int bn, cudaStream_t st)
{
    constexpr int kBlk = KB;
    constexpr int kABytes = kBlk * 2048;
    static PsgDeviceOnce attr_once;
    if (attr_once.need()) {
        if (cudaFuncSetAttribute(gemm_tc_kernel<EPI, X3, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess)
            return PSG_ECUDA;
        attr_once.mark();
    }
    const int stage_bytes = (X3 ? 2 : 1) * (kABytes + kBlk * bn * 16);
    int nst = kRingBytes / stage_bytes;
    if (nst > kMaxStages) nst = kMaxStages;
    // a short K loop needs no deeper ring than it has stages: the narrow layers (K = 16 .. 128, thousands of row tiles)
    // then fit several CTAs per SM instead of one behind a 200 KB ring, and their prologues overlap
    const int kstages = (g.k1chunks + kBlk - 1) / kBlk + (g.k2chunks + kBlk - 1) / kBlk;
    if (nst > kstages) nst = kstages;
    // many tiles and a long K loop: three stages per CTA so that TWO CTAs share an SM -- one's epilogue and prologue run
    // under the other's K loop (a single CTA behind the whole ring serialises them: MSG sa4, 256 row tiles x K = 512)
    if (!X3 && KB == 8 && nst > kNstPlain) nst = kNstPlain;
    if (X3 && bn <= 64 && nst > kNstX3 && (long long)g.mtiles * ((g.nout_pad + bn - 1) / bn) > kBigCtas) nst = kNstX3;
    const size_t smem = (size_t)nst * stage_bytes + 1024;
    dim3 grid((unsigned)g.mtiles, (unsigned)((g.nout_pad + bn - 1) / bn));
    // weights [K/4][Nw][4] as a tiled TMA source: boxes of kBlk planes x bn columns (K is a multiple of 16, i.e. of
    // 4 planes; a last short stage reads past the layer's planes only if K % 32 != 0, where the map clips)
    CUtensorMap wmap;
    memset(&wmap, 0, sizeof(wmap));
    const long long planes = g.k1chunks + g.k2chunks;
    const int use_map = (!X3 && planes % kBlk == 0 && psg_weight_tmap(&wmap, g.W, planes, g.Nw, kBlk, bn)) ? 1 : 0;
    if (psg_launch_pdl(gemm_tc_kernel<EPI, X3, KB>, grid, dim3(kThreads), smem, st, 1, g, bn, nst, psg_tile_trace_slot(), wmap, use_map) != cudaSuccess) return PSG_ECUDA;
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

template <int EPI, bool X3>
int launch(const PsgGemmArgs &g, cudaStream_t st)
{
    // few row tiles (the deep levels): narrower column tiles spread the layer over more SMs, and the smaller
    // B stages let more of the K loop be in flight at once
    int bn = kBNMax;
    while (bn > 32 && g.mtiles * ((g.nout_pad + bn - 1) / bn) < 96) bn >>= 1;
    if (X3) {
        // 3xTF32 stages hold A, A_lo, W_hi and W_lo: with 128-column tiles one CTA fills an SM.  Layers with far more
        // tiles than SMs take 64-column tiles and a two-stage ring instead, so that two CTAs overlap on every SM.
        if (bn > 64 && (long long)g.mtiles * ((g.nout_pad + bn - 1) / bn) > kBigCtas) bn = 64;
        return launch_kb<EPI, X3, 8>(g, bn, st);
    }
    // 32 KB activation stages by default (the producer's per-stage cost bounds the K loop); 16 KB stages x 3 when the
    // layer has far more tiles than SMs and its ring would otherwise leave one CTA per SM
    const long long ctas = (long long)g.mtiles * ((g.nout_pad + bn - 1) / bn);
    const int kstages16 = (g.k1chunks + 15) / 16 + (g.k2chunks + 15) / 16;
    const long long ring16 = (long long)(kstages16 < kRingBytes / (32768 + 16 * bn * 16) ? kstages16 : kRingBytes / (32768 + 16 * bn * 16)) * (32768 + 16 * bn * 16);
    if (ctas > kBigCtas && ring16 > 112 * 1024) return launch_kb<EPI, false, 8>(g, bn, st);
    return launch_kb<EPI, false, 16>(g, bn, st);
}

}  // namespace

int psg_gemm_tc(const PsgGemmArgs &g, cudaStream_t st)
{
    if (g.k1chunks % 4 || g.k2chunks % 4 || g.k1chunks <= 0 || g.mtiles <= 0 || g.nout_pad % 16) return PSG_EINVAL;
    if (g.Nw < g.nout_pad) return PSG_EINVAL;
    if (g.Wlo) {
        switch (g.epi) {
        case PSG_EPI_BIAS_RELU: return launch<PSG_EPI_BIAS_RELU, true>(g, st);
        case PSG_EPI_BIAS: return launch<PSG_EPI_BIAS, true>(g, st);
        case PSG_EPI_MASK: return launch<PSG_EPI_MASK, true>(g, st);
        case PSG_EPI_NONE: return launch<PSG_EPI_NONE, true>(g, st);
        }
        return PSG_EINVAL;
    }
    switch (g.epi) {
    case PSG_EPI_BIAS_RELU: return launch<PSG_EPI_BIAS_RELU, false>(g, st);
    case PSG_EPI_BIAS: return launch<PSG_EPI_BIAS, false>(g, st);
    case PSG_EPI_MASK: return launch<PSG_EPI_MASK, false>(g, st);
    case PSG_EPI_NONE: return launch<PSG_EPI_NONE, false>(g, st);
    }
    return PSG_EINVAL;
}
