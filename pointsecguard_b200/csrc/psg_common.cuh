// psg_common.cuh -- shared device/host helpers of libpsg_b200 (sm_100a only).
//
// HBM layout of every activation tensor ("T-layout"): rows are points (or (centroid, neighbour)
// pairs), channels are padded to a multiple of 16 and stored as 16-byte chunks, tiled by 128 rows:
//
//     float T[M/128][C/4][128][4]            element (r, k) -> ((r>>7)*(C>>2) + (k>>2))*512 + (r&127)*4 + (k&3)
//
// A 128-row x 4-column chunk plane is 2048 contiguous bytes; this is exactly the K-major,
// no-swizzle UMMA canonical layout (8x16B core matrices, SBO = 128 B, LBO = 2048 B), so a GEMM
// operand tile is a run of whole planes (one bulk copy per plane group) and an epilogue in which
// thread r owns row r writes perfectly coalesced 16-byte pieces.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PSG_OK 0
#define PSG_EINVAL (-1)
#define PSG_EUNSUPPORTED (-2)
#define PSG_EWORKSPACE (-3)
#define PSG_ECUDA (-4)

#define PSG_TILE_M 128

struct TView {
    float *base;   // start of the tensor
    int wchunks;   // padded width / 4
    int c0;        // first chunk of the viewed column slice
};

__host__ __device__ __forceinline__ size_t tv_off(const TView &v, long long row, int chunk)
{
    return ((size_t)(row >> 7) * v.wchunks + v.c0 + chunk) * 512 + (size_t)(row & 127) * 4;
}
__device__ __forceinline__ float4 tv_ld(const TView &v, long long row, int chunk)
{
    return *reinterpret_cast<const float4 *>(v.base + tv_off(v, row, chunk));
}
__device__ __forceinline__ void tv_st(const TView &v, long long row, int chunk, float4 x)
{
    *reinterpret_cast<float4 *>(v.base + tv_off(v, row, chunk)) = x;
}

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline long long round_up_ll(long long x, long long m) { return (x + m - 1) / m * m; }
static inline size_t tl_bytes(long long rows, int cpad) { return (size_t)round_up_ll(rows, 128) * cpad * sizeof(float); }

extern long long g_psg_launch_count;   // kernels launched by this library (net.cu)

// Function attributes (the opt-in to > 48 KB of dynamic shared memory) are per device: one flag per kernel, one bit
// per device ordinal; setting an attribute twice from racing threads is harmless, so an atomic bit mask is enough.
struct PsgDeviceOnce {
    unsigned long long done[2] = {0, 0};          // device ordinals 0..127
    bool need() const
    {
        int d = 0;
        cudaGetDevice(&d);
        return !((__atomic_load_n(&done[(d >> 6) & 1], __ATOMIC_ACQUIRE) >> (d & 63)) & 1ull);
    }
    void mark()
    {
        int d = 0;
        cudaGetDevice(&d);
        __atomic_fetch_or(&done[(d >> 6) & 1], 1ull << (d & 63), __ATOMIC_RELEASE);
    }
};

#define PSG_LAUNCH_CHECK()                                      \
    do {                                                        \
        cudaError_t e__ = cudaGetLastError();                   \
        if (e__ != cudaSuccess) return PSG_ECUDA;               \
        ++g_psg_launch_count;                                   \
    } while (0)

// ---- oracle-exact distance arithmetic (SURVEY.md Appendix B) ---------------------------------
// |p|^2 as torch.sum(p ** 2, -1): separately rounded products, left-to-right adds.
__device__ __forceinline__ float psg_sqnorm(float x, float y, float z)
{
    return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}
// square_distance element: ((-2 * dot) + |src|^2) + |dst|^2 with dot = fma(z,z', fma(y,y', x*x')).
__device__ __forceinline__ float psg_sqdist(float sx, float sy, float sz, float sn,
                                            float dx, float dy, float dz, float dn)
{
    float dot = __fmul_rn(sx, dx);
    dot = __fmaf_rn(sy, dy, dot);
    dot = __fmaf_rn(sz, dz, dot);
    return __fadd_rn(__fadd_rn(__fmul_rn(-2.0f, dot), sn), dn);
}
// FPS distance: ((dx*dx + dy*dy) + dz*dz), no contraction.
__device__ __forceinline__ float psg_fpsdist(float px, float py, float pz, float cx, float cy, float cz)
{
    float dx = __fsub_rn(px, cx), dy = __fsub_rn(py, cy), dz = __fsub_rn(pz, cz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Launch with programmatic stream serialization (and optionally a cluster dimension).  Kernels launched
// this way MUST execute griddepcontrol.wait in every CTA before touching data written by earlier kernels.
template <class... KArgs, class... Args>
static inline cudaError_t psg_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster,
                                         Args &&...args)
{
    cudaLaunchConfig_t cfg;
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
    if (cluster > 1) {
        at[na].id = cudaLaunchAttributeClusterDimension;
        at[na].val.clusterDim.x = (unsigned)cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg.attrs = at; cfg.numAttrs = (unsigned)na;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
