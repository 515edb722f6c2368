// fps.cu -- farthest point sampling (reference: PointNet/models/pointnet_util.py:63-84).
//
// One persistent CTA per problem (= one cloud of one forward pass).  The running min-distance
// lives in registers, the cloud in registers + shared memory, and each of the npoint dependent
// rounds costs ONE block barrier: a per-thread scan, two warp REDUX instructions (max of the
// distance bits, then min index among the maxima = torch.max's first-max tie-break), one shared
// write per warp, the barrier, and a second REDUX pair that every warp performs redundantly on the
// 32 per-warp candidates.  Distances use the oracle's exact op order (no FMA).
//
// Many problems (blocks x attack iterations) are launched at once, which is what turns the
// latency-bound recurrence into a throughput problem on 148 SMs (SURVEY.md finding 2).
#include "psg_common.cuh"
#include "psg_internal.h"

namespace {

constexpr int kIntMax = 0x7fffffff;

__device__ __forceinline__ void warp_argmax(unsigned &bits, int &idx)
{
    unsigned m = __reduce_max_sync(0xffffffffu, bits);
    int cand = (bits == m) ? idx : kIntMax;
    idx = __reduce_min_sync(0xffffffffu, cand);
    bits = m;
}

// Packed fp32x2 arithmetic (FADD2 / FFMA2 on sm_100a): two points per instruction for the three subtractions and
// the three squares, each half rounded exactly like the scalar op.  The two ADDS stay scalar on purpose: ptxas
// contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (seen in SASS, even with explicit .rn), which would change
// the rounding; a scalar FADD of one half of a packed product is never contracted (checked in SASS: no FFMA2 with
// a non-zero addend in this file).
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi)
{
    unsigned long long v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ void f2_unpack(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long f2_sub(unsigned long long a, unsigned long long b)
{
    unsigned long long v;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(v) : "l"(a), "l"(b));
    return v;
}
__device__ __forceinline__ unsigned long long f2_sq(unsigned long long a)
{
    unsigned long long v;
    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(v) : "l"(a));
    return v;
}
// distances of two points (lo, hi halves) to the centroid, op order of psg_fpsdist
__device__ __forceinline__ void fpsdist2(unsigned long long px, unsigned long long py, unsigned long long pz,
                                         unsigned long long cx, unsigned long long cy, unsigned long long cz, float &d0, float &d1)
{
    const unsigned long long sx = f2_sq(f2_sub(px, cx)), sy = f2_sq(f2_sub(py, cy)), sz = f2_sq(f2_sub(pz, cz));
    float x0, x1, y0, y1, z0, z1;
    f2_unpack(sx, x0, x1); f2_unpack(sy, y0, y1); f2_unpack(sz, z0, z1);
    d0 = __fadd_rn(__fadd_rn(x0, y0), z0);
    d1 = __fadd_rn(__fadd_rn(x1, y1), z1);
}

// MODE 0: coordinates in registers (+ shared copy for the centroid broadcast), N <= THREADS*PPT
// MODE 1: coordinates only in shared memory (N <= 16384), min-distance in registers
// EXACT:  N == THREADS*PPT, no bounds checks in the round loop (the common 4096 / 1024 / 256 / 64 case)
//
// The round loop is issue-bound (every round touches every point), so it is written to minimise
// instructions: min-distance update is one FMNMX, the per-thread arg-max keeps (value, slot) with a
// strict '>' (slots ascend with the point index, so the first maximum wins as torch.max does), and
// the point index is formed once per round.
template <int THREADS, int PPT, int MODE, bool EXACT>
__global__ void __launch_bounds__(THREADS)
fps_kernel(const float *__restrict__ xyz, long long cloud_stride, int nclouds, int N, int npoint,
           const int *__restrict__ start, int *__restrict__ out_idx, float *__restrict__ out_xyz)
{
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + N, *sz = smem + 2 * N;
    unsigned *red_v = reinterpret_cast<unsigned *>(smem + 3 * N);   // [2][32]
    int *red_i = reinterpret_cast<int *>(red_v + 64);               // [2][32]

    const int p = blockIdx.x;
    const int t = threadIdx.x;
    const int lane = t & 31, warp = t >> 5;
    constexpr int NW = THREADS / 32;
    const float *cloud = xyz + (long long)(p % nclouds) * cloud_stride;

    constexpr bool PK = (MODE == 0 && PPT % 2 == 0);     // two points per packed register pair
    float px[MODE == 0 ? PPT : 1], py[MODE == 0 ? PPT : 1], pz[MODE == 0 ? PPT : 1];
    unsigned long long qx[PK ? PPT / 2 : 1], qy[PK ? PPT / 2 : 1], qz[PK ? PPT / 2 : 1];
    float mind[PPT];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        int i = k * THREADS + t;
        // slots past the end of the cloud keep -1 (below every real distance): never selected
        mind[k] = (EXACT || i < N) ? 1e10f : -1.f;
        if (EXACT || i < N) {
            float x = cloud[3 * i], y = cloud[3 * i + 1], z = cloud[3 * i + 2];
            sx[i] = x; sy[i] = y; sz[i] = z;
            if (MODE == 0) { px[k] = x; py[k] = y; pz[k] = z; }
        } else if (MODE == 0) { px[k] = py[k] = pz[k] = 0.f; }
    }
    if (PK) {
#pragma unroll
        for (int k = 0; k < PPT / 2; ++k) {
            qx[k] = f2_pack(px[2 * k], px[2 * k + 1]); qy[k] = f2_pack(py[2 * k], py[2 * k + 1]); qz[k] = f2_pack(pz[2 * k], pz[2 * k + 1]);
        }
    }
    int far = start[p];
    __syncthreads();

    int *oi = out_idx + (long long)p * npoint;
    float *ox = out_xyz ? out_xyz + (long long)p * npoint * 3 : nullptr;
    int buf = 0;
    for (int it = 0; it < npoint; ++it) {
        const float cx = sx[far], cy = sy[far], cz = sz[far];
        if (t == 0) {
            oi[it] = far;
            if (ox) { ox[3 * it] = cx; ox[3 * it + 1] = cy; ox[3 * it + 2] = cz; }
        }
        float bestv = -2.f; int bestk = 0;
        if (PK) {
            // slots past the end of a ragged cloud hold (0, 0, 0) and the -1 sentinel: fminf(-1, d >= 0) keeps it
            const unsigned long long c2x = f2_pack(cx, cx), c2y = f2_pack(cy, cy), c2z = f2_pack(cz, cz);
#pragma unroll
            for (int k = 0; k < PPT / 2; ++k) {
                float d0, d1;
                fpsdist2(qx[k], qy[k], qz[k], c2x, c2y, c2z, d0, d1);
                mind[2 * k] = fminf(mind[2 * k], d0);
                mind[2 * k + 1] = fminf(mind[2 * k + 1], d1);
                if (mind[2 * k] > bestv) { bestv = mind[2 * k]; bestk = 2 * k; }
                if (mind[2 * k + 1] > bestv) { bestv = mind[2 * k + 1]; bestk = 2 * k + 1; }
            }
        } else
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int i = k * THREADS + t;
            if (EXACT || i < N) {
                const float d = (MODE == 0) ? psg_fpsdist(px[k], py[k], pz[k], cx, cy, cz)
                                            : psg_fpsdist(sx[i], sy[i], sz[i], cx, cy, cz);
                mind[k] = fminf(mind[k], d);          // d is never NaN for finite inputs
            }
            if (mind[k] > bestv) { bestv = mind[k]; bestk = k; }
        }
        // distances are >= 0 (or the -1 sentinel, mapped to 0 bits below) so their bit patterns order like unsigned ints
        unsigned best = bestv < 0.f ? 0u : __float_as_uint(bestv);
        int besti = bestv < 0.f ? kIntMax : bestk * THREADS + t;
        warp_argmax(best, besti);
        if (NW > 1) {
            if (lane == 0) { red_v[buf * 32 + warp] = best; red_i[buf * 32 + warp] = besti; }
            __syncthreads();
            best = lane < NW ? red_v[buf * 32 + lane] : 0u;
            besti = lane < NW ? red_i[buf * 32 + lane] : kIntMax;
            warp_argmax(best, besti);
            buf ^= 1;
        }
        far = besti;
    }
}

// Large clouds (16384 < N <= CS * 1024 * PPT): one thread-block CLUSTER per problem.  CTA q of the cluster keeps its
// share of the cloud in registers (running min-distance, packed coordinates) and in shared memory (for the look-up of
// its winner's coordinates); per round every CTA finds its local first arg-max exactly as fps_kernel does, publishes
// (distance bits, index, x, y, z) into a slot of EVERY CTA's shared memory with st.async stores that complete
// transaction bytes on the DESTINATION's mbarrier, and every CTA waits on its own mbarrier only and reduces the CS
// records itself -- no global memory and no cluster-wide barrier on the round's critical path (a barrier.cluster per
// round measured ~1400 of the round's 2400 cycles).  Records and mbarriers are double-buffered by round parity: a CTA
// can run at most one round ahead of a peer (it needs the peer's record of the previous round to finish it), so it
// never writes a buffer the peer still reads.  The single-CTA fallback below re-reads the whole
// cloud from L2 every round (measured L2-bound at ~7 TB/s with 80 problems of 65536 points in flight).
template <int CS, int PPT>
__global__ void __launch_bounds__(1024, 1)
fps_cluster_kernel(const float *__restrict__ xyz, long long cloud_stride, int nclouds, int N, int npoint,
                   const int *__restrict__ start, int *__restrict__ out_idx, float *__restrict__ out_xyz)
{
    static_assert(PPT % 2 == 0, "points are processed in packed pairs");
    constexpr int T = 1024;
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + T * PPT, *sz = smem + 2 * T * PPT;        // this CTA's points, slot = k * T + t
    __shared__ unsigned red_v[2][32];
    __shared__ int red_i[2][32];
    __shared__ __align__(16) float rec[2][CS][8];                            // per parity, per source CTA: bits, idx, x, y, z
    __shared__ __align__(8) unsigned long long rbar[2];                      // per parity: 1 arrival + CS * 32 transaction bytes
    unsigned q;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(q));
    const int p = blockIdx.x / CS;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float *cloud = xyz + (long long)(p % nclouds) * cloud_stride;

    float mind[PPT];
    unsigned long long qx[PPT / 2], qy[PPT / 2], qz[PPT / 2];
    {
        float px[PPT], py[PPT], pz[PPT];
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int i = k * (CS * T) + (int)q * T + t;          // global point index of slot (k, t) of CTA q
            const bool in = i < N;
            px[k] = in ? cloud[3 * i] : 0.f; py[k] = in ? cloud[3 * i + 1] : 0.f; pz[k] = in ? cloud[3 * i + 2] : 0.f;
            mind[k] = in ? 1e10f : -1.f;                          // -1: below every real distance, never selected
            sx[k * T + t] = px[k]; sy[k * T + t] = py[k]; sz[k * T + t] = pz[k];
        }
#pragma unroll
        for (int k = 0; k < PPT / 2; ++k) {
            qx[k] = f2_pack(px[2 * k], px[2 * k + 1]); qy[k] = f2_pack(py[2 * k], py[2 * k + 1]); qz[k] = f2_pack(pz[2 * k], pz[2 * k + 1]);
        }
    }
    int far = start[p];
    float cx = cloud[3 * far], cy = cloud[3 * far + 1], cz = cloud[3 * far + 2];
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&rbar[0]);
    if (t == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");   // every CTA of the cluster is resident before
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");     // anyone writes into a peer's shared memory

    int *oi = out_idx + (long long)p * npoint;
    float *ox = out_xyz ? out_xyz + (long long)p * npoint * 3 : nullptr;
    for (int it = 0; it < npoint; ++it) {
        const int par = it & 1;
        if (q == 0 && t == 0) {
            oi[it] = far;
            if (ox) { ox[3 * it] = cx; ox[3 * it + 1] = cy; ox[3 * it + 2] = cz; }
        }
        float bestv = -2.f; int bestk = 0;
        const unsigned long long c2x = f2_pack(cx, cx), c2y = f2_pack(cy, cy), c2z = f2_pack(cz, cz);
#pragma unroll
        for (int k = 0; k < PPT / 2; ++k) {
            float d0, d1;
            fpsdist2(qx[k], qy[k], qz[k], c2x, c2y, c2z, d0, d1);
            mind[2 * k] = fminf(mind[2 * k], d0);
            mind[2 * k + 1] = fminf(mind[2 * k + 1], d1);
            // slots ascend with the global index inside a thread (k major), so strict '>' keeps the first maximum
            if (mind[2 * k] > bestv) { bestv = mind[2 * k]; bestk = 2 * k; }
            if (mind[2 * k + 1] > bestv) { bestv = mind[2 * k + 1]; bestk = 2 * k + 1; }
        }
        unsigned best = bestv < 0.f ? 0u : __float_as_uint(bestv);
        int besti = bestv < 0.f ? kIntMax : bestk * (CS * T) + (int)q * T + t;
        warp_argmax(best, besti);
        if (lane == 0) { red_v[par][warp] = best; red_i[par][warp] = besti; }
        __syncthreads();
        if (warp == 0) {
            best = red_v[par][lane]; besti = red_i[par][lane];
            warp_argmax(best, besti);
            // the CTA's candidate and its coordinates -> slot q of every CTA's record table
            float bx = 0.f, by = 0.f, bz = 0.f;
            if (besti != kIntMax) {
                const int slot = (besti / (CS * T)) * T + (besti % T);
                bx = sx[slot]; by = sy[slot]; bz = sz[slot];
            }
            if (lane == 0)            // this round's phase of OUR barrier completes when this arrival and all CS records are in
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8u * par), "r"((uint32_t)CS * 32u) : "memory");
            if (lane < CS) {
                const uint32_t local = (uint32_t)__cvta_generic_to_shared(&rec[par][q][0]);
                uint32_t remote, rbar_remote;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"((uint32_t)lane));
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar_remote) : "r"(bar0 + 8u * par), "r"((uint32_t)lane));
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(remote),
                             "r"(best), "r"((unsigned)besti), "r"(__float_as_uint(bx)), "r"(__float_as_uint(by)), "r"(rbar_remote) : "memory");
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(remote + 16u),
                             "r"(__float_as_uint(bz)), "r"(0u), "r"(0u), "r"(0u), "r"(rbar_remote) : "memory");
            }
        }
        {
            // wait for this round's CS records (phase parity of barrier `par` flips every second round)
            const uint32_t ph = (uint32_t)(it >> 1) & 1u, bar = bar0 + 8u * par;
            uint32_t ok;
            do {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(ok) : "r"(bar), "r"(ph) : "memory");
            } while (!ok);
        }
        // every warp reduces the CS records redundantly (first maximum = smallest index among equal distances)
        {
            const float4 r4 = lane < CS ? *reinterpret_cast<const float4 *>(&rec[par][lane][0]) : make_float4(0.f, __int_as_float(kIntMax), 0.f, 0.f);
            const float rz = lane < CS ? rec[par][lane][4] : 0.f;
            unsigned b = __float_as_uint(r4.x); int bi = __float_as_int(r4.y);
            const int mine = bi;
            warp_argmax(b, bi);
            const unsigned win = __ballot_sync(0xffffffffu, mine == bi && lane < CS);
            const int src = __ffs(win) - 1;
            far = bi;
            cx = __shfl_sync(0xffffffffu, r4.z, src); cy = __shfl_sync(0xffffffffu, r4.w, src); cz = __shfl_sync(0xffffffffu, rz, src);
        }
    }
    // no CTA may exit while a peer can still write into its shared memory
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Fallback for clouds that fit neither registers nor shared memory (N > 16384): coordinates are
// re-read from L2 every round and the min-distance lives in a caller-provided workspace.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
fps_global_kernel(const float *__restrict__ xyz, long long cloud_stride, int nclouds, int N, int npoint,
                  const int *__restrict__ start, int *__restrict__ out_idx, float *__restrict__ out_xyz,
                  float *__restrict__ mind_ws)
{
    __shared__ unsigned red_v[64];
    __shared__ int red_i[64];
    const int p = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    constexpr int NW = THREADS / 32;
    const float *cloud = xyz + (long long)(p % nclouds) * cloud_stride;
    float *mind = mind_ws + (long long)p * N;
    for (int i = t; i < N; i += THREADS) mind[i] = 1e10f;
    int far = start[p];
    int buf = 0;
    for (int it = 0; it < npoint; ++it) {
        const float cx = cloud[3 * far], cy = cloud[3 * far + 1], cz = cloud[3 * far + 2];
        if (t == 0) {
            out_idx[(long long)p * npoint + it] = far;
            if (out_xyz) {
                float *o = out_xyz + ((long long)p * npoint + it) * 3;
                o[0] = cx; o[1] = cy; o[2] = cz;
            }
        }
        unsigned best = 0u; int besti = kIntMax;
        for (int i = t; i < N; i += THREADS) {
            float d = psg_fpsdist(cloud[3 * i], cloud[3 * i + 1], cloud[3 * i + 2], cx, cy, cz);
            float m = mind[i];
            if (d < m) { m = d; mind[i] = d; }
            unsigned b = __float_as_uint(m);
            if (b > best || besti == kIntMax) { best = b; besti = i; }
        }
        warp_argmax(best, besti);
        if (lane == 0) { red_v[buf * 32 + warp] = best; red_i[buf * 32 + warp] = besti; }
        __syncthreads();
        best = lane < NW ? red_v[buf * 32 + lane] : 0u;
        besti = lane < NW ? red_i[buf * 32 + lane] : kIntMax;
        warp_argmax(best, besti);
        buf ^= 1;
        far = besti;
    }
}

template <int THREADS, int PPT, int MODE>
int launch_fps(const float *xyz, long long cloud_stride, int nclouds, int P, int N, int npoint,
               const int *start, int *out_idx, float *out_xyz, cudaStream_t st)
{
    size_t smem = (size_t)3 * N * sizeof(float) + 128 * sizeof(int);
    auto kern = (N == THREADS * PPT) ? fps_kernel<THREADS, PPT, MODE, true> : fps_kernel<THREADS, PPT, MODE, false>;
    if (smem > 48 * 1024) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return PSG_ECUDA;
    }
    // several problems share an SM (that is what hides the per-round reduction latency): ask for the largest
    // shared-memory carve-out so that the clouds of three or four CTAs fit next to each other
    if (cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess)
        return PSG_ECUDA;
    kern<<<P, THREADS, smem, st>>>(xyz, cloud_stride, nclouds, N, npoint, start, out_idx, out_xyz);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

}  // namespace

// one CS-CTA cluster per problem; the per-thread share is 2, 4 or 8 points
template <int CS>
static int launch_fps_cluster(int ppt, const float *xyz, long long cloud_stride, int nclouds, int P, int N, int npoint,
                              const int *start, int *out_idx, float *out_xyz, cudaStream_t st)
{
    auto kern = ppt == 2 ? fps_cluster_kernel<CS, 2> : (ppt == 4 ? fps_cluster_kernel<CS, 4> : fps_cluster_kernel<CS, 8>);
    const size_t smem = (size_t)3 * 1024 * ppt * sizeof(float);
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return PSG_ECUDA;
    cudaLaunchConfig_t cfg;
    cfg.gridDim = dim3((unsigned)P * CS); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kern, xyz, cloud_stride, nclouds, N, npoint, start, out_idx, out_xyz) != cudaSuccess) {
        cudaGetLastError();
        return PSG_ECUDA;
    }
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}

// cluster kernels for 16384 < N <= 65536 (and few problems of 8192 < N <= 16384), on by default; psg_set_option
// "fps_cluster" 0 selects the single-CTA kernels, the reference tests/test_gpu_primitives.py matches them against bit for bit
static int g_fps_cluster = 1;
void psg_fps_use_cluster(int on) { g_fps_cluster = on; }

size_t psg_fps_workspace_bytes(int P, int N)
{
    return N > 16384 ? (size_t)P * N * sizeof(float) : 0;
}

int psg_fps_launch(const float *xyz, long long cloud_stride, int nclouds, int P, int N, int npoint,
                   const int *start, int *out_idx, float *out_xyz, void *ws, size_t ws_bytes,
                   cudaStream_t st)
{
    if (P <= 0 || N <= 0 || npoint <= 0 || nclouds <= 0) return PSG_EINVAL;
    if (N <= 64) return launch_fps<64, 1, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (N <= 256) return launch_fps<256, 1, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (N <= 1024) return launch_fps<512, 2, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (N <= 2048) return launch_fps<512, 4, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    // many problems in flight (attack geometry batches): fewer, fatter threads -- the per-round warp
    // overhead (REDUX, barrier, exchange) is amortised over 16 points and 4 CTAs share an SM
    // (from 128 problems on: moving the threshold measured no difference for the smaller geometry passes)
    if (N <= 4096 && N > 2048 && P >= 128)
        return launch_fps<256, 16, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (N <= 4096) return launch_fps<1024, 4, 0>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    // few problems of a medium cloud: a cluster per problem (all resident at once) beats one CTA walking 16 points per
    // thread out of shared memory (1.0 vs 1.5 us per round); with many problems in flight the single CTAs fill the GPU
    if (g_fps_cluster && N > 8192 && N <= 16384 && P * 8 <= 128)
        return launch_fps_cluster<8>(2, xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (N <= 16384) return launch_fps<1024, 16, 1>(xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    if (g_fps_cluster && N <= 8 * 1024 * 8) {
        constexpr int CS = 8;
        const int ppt = N <= CS * 1024 * 2 ? 2 : (N <= CS * 1024 * 4 ? 4 : 8);
        return launch_fps_cluster<CS>(ppt, xyz, cloud_stride, nclouds, P, N, npoint, start, out_idx, out_xyz, st);
    }
    if (ws_bytes < psg_fps_workspace_bytes(P, N) || !ws) return PSG_EWORKSPACE;
    fps_global_kernel<1024><<<P, 1024, 0, st>>>(xyz, cloud_stride, nclouds, N, npoint, start, out_idx, out_xyz,
                                                (float *)ws);
    PSG_LAUNCH_CHECK();
    return PSG_OK;
}
