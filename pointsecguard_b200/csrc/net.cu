// net.cu -- the whole-network engine: PointNet++ sem-seg forward, input-gradient backward and the
// norm-bounded attack loop as plain sequences of kernel launches on one stream.
//
// Reference: PointNet/models/pointnet2_sem_seg.py:22-40, pointnet2_sem_seg_msg.py:23-41 (forward),
// PointNet/models/pointnet_util.py:166-320 (SA / SA-MSG / FP modules), autograd of the same for the
// backward, PointNet/attacks/torchattacks/attacks/nontarget.py:28-39 and target.py:31-43 (loops).
//
// Design (DESIGN.md section 3-4):
//   * Geometry (FPS, ball query, 3-NN, and the source-sorted CSRs the deterministic gather-backward
//     needs) depends only on xyz and on the FPS start draws, so for colour attacks it is computed
//     for all T forwards of an attack in one batched pass (T*B FPS problems fill the 148 SMs) and
//     kept resident as int32 indices + fp32 weights.
//   * Activations live in T-layout (psg_common.cuh); every conv(1x1)+BN(eval)+ReLU is one GEMM with
//     the BN folded into W,b; FP concat is a two-source A operand; dgrad only, no wgrad.
//   * No allocation, no synchronisation, no host round trip inside forward / backward / attack.
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/psg_b200.h"
#include "psg_common.cuh"
#include "psg_internal.h"

long long g_psg_launch_count = 0;
// FP levels with fewer 128-row tiles than this run per layer: with a third of the SMs or fewer busy, 64 column-split
// GEMM CTAs with a deep operand ring beat one cluster per tile (B = 16: fp3 as a tile program 1133 steps/s, per
// layer 1153)
static const int kFpMinTiles = 48;
// fused SA branches run on compacted neighbourhood rows (compact.cu); psg_set_option "sa_compact" 0 restores the padded layout
static int g_sa_compact = 1;
// mode 2 (3xTF32): the narrow SA branches run as fused kernels too when their hi + lo weights and operand buffers fit
// (psg_set_option "x3_fused" 0: every layer of mode 2 goes through the per-layer GEMM)
static int g_x3_fused = 3;     // bit 0: the narrow SA branches, bit 1: fp1 + head

// ------------------------------------------------------------------------------------------------
// per-kernel-family device timing (bench.py's live roofline measurement).  When enabled, every
// launch of the engine is bracketed by a CUDA event pair on the launching stream; collect() syncs
// and sums the elapsed times per family.  Off by default (zero overhead, graph-capture safe).
// ------------------------------------------------------------------------------------------------
enum { PF_FPS, PF_BALL, PF_NN3, PF_CSR, PF_PACK, PF_GROUP, PF_GEMM_FWD, PF_MAXPOOL, PF_INTERP, PF_HEAD, PF_LOSS,
       PF_GEMM_BWD, PF_MAXPOOL_BWD, PF_SEGSUM, PF_COPY, PF_PGD, PF_SA_FWD, PF_SA_BWD, PF_FP_FWD, PF_FP_BWD, PF_HEAD_CHAIN,
       PF_NCAT };
static const char *kProfNames[PF_NCAT] = {"fps", "ball_query", "three_nn", "csr_build", "pack", "group", "gemm_fwd",
                                          "maxpool", "interp", "head", "loss_grad", "gemm_bwd", "maxpool_bwd", "segsum",
                                          "copy_cols", "pgd_update", "sa_fused_fwd", "sa_fused_bwd", "fp_fused_fwd",
                                          "fp_fused_bwd", "head_chain"};
namespace {
struct ProfRec { cudaEvent_t a, b; int cat; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
cudaEvent_t prof_event()
{
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
}
struct ProfScope {
    int cat; cudaStream_t st; cudaEvent_t a; bool on;
    ProfScope(int c, cudaStream_t s) : cat(c), st(s), a(nullptr), on(g_prof_on)
    {
        if (on) { a = prof_event(); cudaEventRecord(a, st); }
    }
    void end()
    {
        if (on) { cudaEvent_t b = prof_event(); cudaEventRecord(b, st); g_prof_recs.push_back(ProfRec{a, b, cat}); }
    }
};
}  // namespace

extern "C" int psg_prof_enable(int on) { g_prof_on = on != 0; return PSG_OK; }
extern "C" int psg_prof_ncat(void) { return PF_NCAT; }
extern "C" const char *psg_prof_name(int cat) { return cat >= 0 && cat < PF_NCAT ? kProfNames[cat] : ""; }
extern "C" int psg_prof_collect(double *ms_by_cat, int64_t *count_by_cat)
{
    if (cudaDeviceSynchronize() != cudaSuccess) return PSG_ECUDA;
    for (int c = 0; c < PF_NCAT; ++c) { if (ms_by_cat) ms_by_cat[c] = 0.0; if (count_by_cat) count_by_cat[c] = 0; }
    for (const ProfRec &r : g_prof_recs) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        if (ms_by_cat) ms_by_cat[r.cat] += ms;
        if (count_by_cat) count_by_cat[r.cat] += 1;
        g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b);
    }
    g_prof_recs.clear();
    return PSG_OK;
}

#define PSG_RUN(cat, call)                \
    do {                                  \
        ProfScope ps__(cat, st);          \
        int rc__ = (call);                \
        ps__.end();                       \
        if (rc__ != PSG_OK) return rc__;  \
    } while (0)

// ------------------------------------------------------------------------------------------------
// one folded layer
// ------------------------------------------------------------------------------------------------
struct psg_mlp {
    int cin, cout;
    int kpad;        // input columns, multiple of 16
    int npad;        // output columns, multiple of 16
    int nwf, nwb;    // packed widths (multiples of 64) of the forward / dgrad weight copies
    float *wf;       // [kpad/4][nwf][4]   wf[(k/4, n, k%4)] = W[n][k]
    float *wb;       // [npad/4][nwb][4]   wb[(n/4, k, n%4)] = W[n][k]
    float *bias;     // [nwf]
    float *wf_tf32, *wb_tf32;   // the same two packings for the tcgen05 path: TF32 values, truncation-compensated (below)
    float *wf_hi, *wf_lo, *wb_hi, *wb_lo;   // mode 2 (3xTF32): W_hi = nearest TF32 of W, W_lo = nearest TF32 of W - W_hi
};

// tcgen05.mma kind::tf32 reads the upper 19 bits of its fp32 operands: it TRUNCATES.  Truncation loses half a TF32 ulp on
// average, -3.5e-4 relative per operand (mean of 2^-11 / mantissa over a log-uniform mantissa), always towards zero, so
// the bias adds up coherently layer after layer: 23 layers x 2 operands = -1.6 % on the logits of the trained network,
// max |d logp| 0.35, 8 % flipped gradient signs -- measured, tools/grad_diag.py.  Both halves are repaired here for free:
//   * the weights are rounded to NEAREST TF32 on the host (the hardware then truncates nothing of them);
//   * the activations' mean truncation loss is folded into the weights as the factor (1 + kTf32Comp) before rounding.
// What remains is zero-mean rounding noise (std ~0.29 ulp per operand, the same as round-to-nearest would leave), which
// averages over the K terms of a dot product instead of accumulating.
static const double kTf32Comp = 3.45e-4;
static const double kX3AccComp = 6.6e-9;       // 3xTF32 accumulator truncation per column of contraction (psg_mlp_create)
static inline float tf32_rna(double x)
{
    float f = (float)x;
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7f800000u) != 0x7f800000u) u = (u + 0x1000u) & 0xffffe000u;
    memcpy(&f, &u, 4);
    return f;
}
static inline const float *w_fwd(const psg_mlp *m, int mode) { return mode == 1 ? m->wf_tf32 : mode == 2 ? m->wf_hi : m->wf; }
static inline const float *w_bwd(const psg_mlp *m, int mode) { return mode == 1 ? m->wb_tf32 : mode == 2 ? m->wb_hi : m->wb; }

extern "C" psg_mlp *psg_mlp_create(const float *w, const float *b, int cin, int cout)
{
    if (!w || cin <= 0 || cout <= 0) return nullptr;
    psg_mlp *m = new (std::nothrow) psg_mlp();
    if (!m) return nullptr;
    m->cin = cin; m->cout = cout;
    m->kpad = round_up(cin, 16);
    m->npad = round_up(cout, 16);
    m->nwf = round_up(m->npad, 64);
    m->nwb = round_up(m->kpad, 64);
    std::vector<float> hf((size_t)m->kpad * m->nwf, 0.f), hb((size_t)m->npad * m->nwb, 0.f), hbias(m->nwf, 0.f);
    for (int n = 0; n < cout; ++n) {
        for (int k = 0; k < cin; ++k) {
            const float v = w[(size_t)n * cin + k];
            hf[((size_t)(k >> 2) * m->nwf + n) * 4 + (k & 3)] = v;
            hb[((size_t)(n >> 2) * m->nwb + k) * 4 + (n & 3)] = v;
        }
        hbias[n] = b ? b[n] : 0.f;
    }
    m->wf = m->wb = m->bias = m->wf_tf32 = m->wb_tf32 = nullptr;
    m->wf_hi = m->wf_lo = m->wb_hi = m->wb_lo = nullptr;
    std::vector<float> cf(hf.size()), cb(hb.size());
    for (size_t i = 0; i < hf.size(); ++i) cf[i] = tf32_rna((double)hf[i] * (1.0 + kTf32Comp));
    for (size_t i = 0; i < hb.size(); ++i) cb[i] = tf32_rna((double)hb[i] * (1.0 + kTf32Comp));
    // 3xTF32 split of the exact weights (both parts TF32-representable: the hardware's truncation leaves them alone)
    std::vector<float> fh(hf.size()), fl(hf.size()), bh(hb.size()), bl(hb.size());
    // The tensor core's fp32 accumulator TRUNCATES every add (three per 8-column K step in 3xTF32): a layer's output comes
    // out scaled by 1 - 6.6e-9 K (measured, tools/gemm_precision.py: -8.8e-7 at K = 128, -4.8e-6 at K = 768; the random part
    // of the same truncation is half as large).  Like the TF32 mode's operand truncation, the systematic part is folded
    // into the weights: contraction length K = kpad forward, npad in the dgrad.
    const double cf3 = 1.0 + kX3AccComp * m->kpad, cb3 = 1.0 + kX3AccComp * m->npad;
    for (size_t i = 0; i < hf.size(); ++i) { const double v = (double)hf[i] * cf3; fh[i] = tf32_rna(v); fl[i] = tf32_rna(v - (double)fh[i]); }
    for (size_t i = 0; i < hb.size(); ++i) { const double v = (double)hb[i] * cb3; bh[i] = tf32_rna(v); bl[i] = tf32_rna(v - (double)bh[i]); }
    bool ok = cudaMalloc(&m->wf, hf.size() * 4) == cudaSuccess && cudaMalloc(&m->wb, hb.size() * 4) == cudaSuccess &&
              cudaMalloc(&m->wf_tf32, hf.size() * 4) == cudaSuccess && cudaMalloc(&m->wb_tf32, hb.size() * 4) == cudaSuccess &&
              cudaMalloc(&m->bias, hbias.size() * 4) == cudaSuccess &&
              cudaMalloc(&m->wf_hi, hf.size() * 4) == cudaSuccess && cudaMalloc(&m->wf_lo, hf.size() * 4) == cudaSuccess &&
              cudaMalloc(&m->wb_hi, hb.size() * 4) == cudaSuccess && cudaMalloc(&m->wb_lo, hb.size() * 4) == cudaSuccess;
    ok = ok && cudaMemcpy(m->wf_hi, fh.data(), fh.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wf_lo, fl.data(), fl.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wb_hi, bh.data(), bh.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wb_lo, bl.data(), bl.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(m->wf, hf.data(), hf.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wb, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wf_tf32, cf.data(), cf.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->wb_tf32, cb.data(), cb.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(m->bias, hbias.data(), hbias.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok) { psg_mlp_destroy(m); return nullptr; }
    return m;
}

// training: a layer whose weights live in device memory (nn.Parameter storage) and change every optimiser step
extern "C" psg_mlp *psg_mlp_create_device(int cin, int cout)
{
    if (cin <= 0 || cout <= 0) return nullptr;
    psg_mlp *m = new (std::nothrow) psg_mlp();
    if (!m) return nullptr;
    m->cin = cin; m->cout = cout;
    m->kpad = round_up(cin, 16);
    m->npad = round_up(cout, 16);
    m->nwf = round_up(m->npad, 64);
    m->nwb = round_up(m->kpad, 64);
    m->wf = m->wb = m->bias = m->wf_tf32 = m->wb_tf32 = nullptr;
    m->wf_hi = m->wf_lo = m->wb_hi = m->wb_lo = nullptr;       // training layers: modes 0 / 1 only
    const size_t nf = (size_t)m->kpad * m->nwf * 4, nb = (size_t)m->npad * m->nwb * 4;
    bool ok = cudaMalloc(&m->wf, nf) == cudaSuccess && cudaMalloc(&m->wb, nb) == cudaSuccess &&
              cudaMalloc(&m->wf_tf32, nf) == cudaSuccess && cudaMalloc(&m->wb_tf32, nb) == cudaSuccess &&
              cudaMalloc(&m->bias, (size_t)m->nwf * 4) == cudaSuccess;
    if (!ok) { psg_mlp_destroy(m); return nullptr; }
    return m;
}

// (re)pack W [cout][cin] row-major and b [cout] (device memory) into the layer's operand layouts; enqueued on stream
extern "C" int psg_mlp_load(psg_mlp *m, const float *w_dev, const float *b_dev, psg_stream_t stream)
{
    if (!m || !w_dev) return PSG_EINVAL;
    return psg_repack_weights(w_dev, b_dev, m->cout, m->cin, m->kpad, m->npad, m->nwf, m->nwb, m->wf, m->wb, m->wf_tf32,
                              m->wb_tf32, m->bias, (float)kTf32Comp, (cudaStream_t)stream);
}

extern "C" void psg_mlp_destroy(psg_mlp *m)
{
    if (!m) return;
    cudaFree(m->wf); cudaFree(m->wb); cudaFree(m->bias); cudaFree(m->wf_tf32); cudaFree(m->wb_tf32);
    cudaFree(m->wf_hi); cudaFree(m->wf_lo); cudaFree(m->wb_hi); cudaFree(m->wb_lo);
    delete m;
}

static int run_gemm(const PsgGemmArgs &g, int mode, cudaStream_t st)
{
    return mode >= 1 ? psg_gemm_tc(g, st) : psg_gemm_simt(g, st);
}

// forward of one layer: Out = act([A1 | A2] W^T + b)
static int mlp_fwd(const psg_mlp *m, TView a1, int k1chunks, TView a2, int k2chunks, long long rows, TView out,
                   int relu, int mode, cudaStream_t st)
{
    if ((k1chunks + k2chunks) * 4 != m->kpad) return PSG_EINVAL;
    PsgGemmArgs g;
    g.A1 = a1; g.k1chunks = k1chunks; g.A2 = a2; g.k2chunks = k2chunks;
    if (mode == 2 && !m->wf_hi) return PSG_EUNSUPPORTED;
    g.W = w_fwd(m, mode); g.Wlo = mode == 2 ? m->wf_lo : nullptr; g.Nw = m->nwf; g.bias = m->bias; g.Out = out; g.nout_pad = m->npad;
    g.Mask = TView{nullptr, 0, 0};
    g.Out2 = TView{nullptr, 0, 0}; g.out2_cols = 0;
    g.mtiles = (int)(round_up_ll(rows, 128) / 128);
    g.epi = relu ? PSG_EPI_BIAS_RELU : PSG_EPI_BIAS;
    return run_gemm(g, mode, st);
}

// dgrad of one layer: dX = (dY W) [. (mask > 0)]
static int mlp_bwd(const psg_mlp *m, TView dy, long long rows, TView dx, const TView *mask, int mode, cudaStream_t st,
                   const TView *out2 = nullptr, int out2_cols = 0)
{
    PsgGemmArgs g;
    g.Out2 = out2 ? *out2 : TView{nullptr, 0, 0}; g.out2_cols = out2 ? out2_cols : 0;
    g.A1 = dy; g.k1chunks = m->npad / 4; g.A2 = TView{nullptr, 0, 0}; g.k2chunks = 0;
    if (mode == 2 && !m->wb_hi) return PSG_EUNSUPPORTED;
    g.W = w_bwd(m, mode); g.Wlo = mode == 2 ? m->wb_lo : nullptr; g.Nw = m->nwb; g.bias = nullptr; g.Out = dx; g.nout_pad = m->kpad;
    g.Mask = mask ? *mask : TView{nullptr, 0, 0};
    g.mtiles = (int)(round_up_ll(rows, 128) / 128);
    g.epi = mask ? PSG_EPI_MASK : PSG_EPI_NONE;
    return run_gemm(g, mode, st);
}

extern "C" int psg_mlp_forward(const psg_mlp *m, const float *a1_base, int a1_wchunks, int a1_c0, int k1chunks,
                               const float *a2_base, int a2_wchunks, int a2_c0, int k2chunks, int64_t rows,
                               float *out_base, int out_wchunks, int relu, int mode, psg_stream_t stream)
{
    if (!m || !a1_base || !out_base || rows <= 0) return PSG_EINVAL;
    return mlp_fwd(m, TView{(float *)a1_base, a1_wchunks, a1_c0}, k1chunks, TView{(float *)a2_base, a2_wchunks, a2_c0},
                   k2chunks, rows, TView{out_base, out_wchunks, 0}, relu, mode, (cudaStream_t)stream);
}

extern "C" int psg_mlp_backward(const psg_mlp *m, const float *dy_base, int dy_wchunks, int64_t rows, float *dx_base,
                                int dx_wchunks, const float *mask_base, int mask_wchunks, int mode, psg_stream_t stream)
{
    if (!m || !dy_base || !dx_base || rows <= 0) return PSG_EINVAL;
    TView mk{(float *)mask_base, mask_wchunks, 0};
    return mlp_bwd(m, TView{(float *)dy_base, dy_wchunks, 0}, rows, TView{dx_base, dx_wchunks, 0},
                   mask_base ? &mk : nullptr, mode, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// the network
// ------------------------------------------------------------------------------------------------
namespace {

struct Bump {
    char *base;
    size_t off;
    template <class T> T *take(size_t n)
    {
        off = (off + 1023) & ~(size_t)1023;
        T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += n * sizeof(T);
        return p;
    }
    float *tl(long long rows, int cpad) { return take<float>(tl_bytes(rows, cpad) / sizeof(float)); }
};

struct Branch {
    int K, nl;
    psg_mlp *mlp[3];
    int gpad;              // padded width of the grouped input (D + 3 -> multiple of 16)
    int col0;              // first output column inside the level's feature tensor
    float *G, *Y[3];
    unsigned char *arg;
    int *ball;             // [T*B][S][K]
    bool fused;            // tcgen05 mode runs the branch as one kernel per direction (sa_fused.cu)
    bool streamed;         // ... or, for wide layers, as a tile program with streamed weights (chain_fused.cu)
    unsigned *m0, *m1;     // ReLU bits of layers 0 / 1 (fused path)
    int *csr_off, *csr_perm;   // [T*B][R+1], [T*B][S*K]
    bool compactable;      // fused branch whose kernels can run on compacted rows (real ball-query hits only, compact.cu)
    PsgCompact cp;
};

struct SaLevel {
    int S, nbr;
    double radius[2];
    Branch br[2];
};

struct FpLevel {
    int nl;
    psg_mlp *mlp[3];
    int C1, C2;            // skip width (fine level features), interpolated width (coarse features)
    float *I, *Y[3];
    float *Yrm;            // row-major mirror of the last layer's output (the next finer level gathers from it)
    int *nn_idx;           // [T*B][Nf][3]
    float *nn_w;           // [T*B][Nf][3]
    int *csr_off, *csr_perm;   // [T*B][Nc+1], [T*B][Nf*3]
    bool streamed;         // tcgen05 mode: forward and backward run as tile programs (chain_fused.cu)
    unsigned *m[3];        // ReLU bits of the hidden layers (streamed path)
};

}  // namespace

struct psg_net {
    int in_channels, ncls, mode;
    SaLevel sa[4];
    FpLevel fp[4];
    psg_mlp *conv1, *conv2;
    // bound problem
    int B, N, T;
    int npts[5], cfeat[5], wfeat[5];
    float *xyz0;           // [B][N][3]
    float *xyz[5];         // [T*B][S_l][3], l = 1..4
    int *fps_idx[5];
    int *starts;           // [4][T][B]
    void *fps_ws; size_t fps_ws_bytes;
    void *csr_ws;
    void *grid_ws;         // uniform grid over the level-0 clouds (ballgrid.cu), when N is large
    bool grid_valid;
    float *feats[5], *dfeat[5];
    float *H, *Z, *dZ;
    float *S[2]; size_t scratch_floats;
    float *Srm;            // row-major copy of the gradient rows a fused backward kernel hands to the segmented sum
    bool bound;
    int last_t;
    // tcgen05 mode: fp1 + head run as one forward+backward kernel (chain_fused.cu); the loss is then
    // evaluated inside psg_net_backward from this deferred specification
    bool xyz_grad;         // also produce the geometric gradient w.r.t. coordinates (geomgrad.cu)
    float *dxyz[5];        // [B][npts[l]][3]
    float *xyz_tmp;        // [B][N*3][3] coarse-side vectors of the interpolation backward
    bool head_fused;
    bool compact_valid;    // the resident geometry carries compacted rows for the fused SA branches
    bool z_valid;          // logits of the last forward are materialised in Z
    struct { int kind, target; const float *dlogp; const int *labels; float scale, kappa; float *loss_rows;
             unsigned char *hit; bool set; } loss;
};

static psg_mlp *make_layer(const psg_mlp_desc &d) { return psg_mlp_create(d.w_host, d.b_host, d.cin, d.cout); }

extern "C" psg_net *psg_net_create(const psg_net_desc *d)
{
    if (!d || d->in_channels < 3 || d->in_channels > 16 || d->num_classes < 2 || d->num_classes > 16) return nullptr;
    psg_net *n = new (std::nothrow) psg_net();
    if (!n) return nullptr;
    memset(n, 0, sizeof(*n));
    n->in_channels = d->in_channels; n->ncls = d->num_classes; n->mode = d->mlp_mode;
    bool ok = true;
    int cprev = d->in_channels;
    n->cfeat[0] = cprev; n->wfeat[0] = round_up(cprev, 16);
    for (int l = 0; l < 4 && ok; ++l) {
        const psg_sa_desc &s = d->sa[l];
        SaLevel &L = n->sa[l];
        L.S = s.npoint; L.nbr = s.nbranch;
        if (s.nbranch < 1 || s.nbranch > 2 || s.npoint < 3) { ok = false; break; }
        int col = 0;
        for (int b = 0; b < s.nbranch && ok; ++b) {
            Branch &R = L.br[b];
            L.radius[b] = s.radius[b];
            R.K = s.nsample[b]; R.nl = s.nlayers[b];
            if ((R.K != 16 && R.K != 32) || R.nl < 1 || R.nl > 3) { ok = false; break; }
            R.gpad = round_up(cprev + 3, 16);
            int cin = cprev + 3;
            for (int j = 0; j < R.nl; ++j) {
                if (s.mlp[b][j].cin != cin) { ok = false; break; }
                R.mlp[j] = make_layer(s.mlp[b][j]);
                if (!R.mlp[j]) { ok = false; break; }
                cin = s.mlp[b][j].cout;
            }
            if (!ok) break;
            if (cin % 16) { ok = false; break; }      // branch outputs are concatenated on 16-column boundaries
            R.col0 = col; col += cin;
        }
        cprev = col;
        n->cfeat[l + 1] = col; n->wfeat[l + 1] = col;
    }
    // FP levels: fp[f] has fine level f, coarse level f+1; runs f = 3, 2, 1, 0
    int cup = n->wfeat[4];
    for (int f = 3; f >= 0 && ok; --f) {
        const psg_fp_desc &s = d->fp[f];
        FpLevel &F = n->fp[f];
        F.nl = s.nlayers;
        F.C1 = f > 0 ? n->wfeat[f] : 0;
        F.C2 = cup;
        if (F.nl < 1 || F.nl > 3 || s.mlp[0].cin != F.C1 + F.C2) { ok = false; break; }
        int cin = s.mlp[0].cin;
        for (int j = 0; j < F.nl; ++j) {
            if (s.mlp[j].cin != cin) { ok = false; break; }
            F.mlp[j] = make_layer(s.mlp[j]);
            if (!F.mlp[j]) { ok = false; break; }
            cin = s.mlp[j].cout;
        }
        if (cin % 16) ok = false;
        cup = cin;
    }
    if (ok) {
        n->conv1 = make_layer(d->conv1);
        n->conv2 = make_layer(d->conv2);
        ok = n->conv1 && n->conv2 && d->conv1.cin == cup && d->conv2.cin == d->conv1.cout && d->conv2.cout == n->ncls &&
             d->conv1.cout % 16 == 0;
    }
    if (!ok) { psg_net_destroy(n); return nullptr; }
    {
        const FpLevel &F = n->fp[0];
        bool hf = F.C1 == 0 && F.C2 % 16 == 0 && F.C2 <= 128 && F.nl + 1 <= 4 && n->conv2->npad == 16 &&
                  n->conv2->nwf <= 128 && n->conv2->nwb == n->conv1->npad;
        int kprev = F.C2;
        for (int j = 0; j < F.nl && hf; ++j) {
            hf = F.mlp[j]->npad <= 128 && F.mlp[j]->nwf == F.mlp[j]->npad && F.mlp[j]->nwb == kprev;
            kprev = F.mlp[j]->npad;
        }
        hf = hf && n->conv1->npad <= 128 && n->conv1->nwf == n->conv1->npad && n->conv1->nwb == kprev;
        n->head_fused = hf;
    }
    return n;
}

extern "C" void psg_net_destroy(psg_net *n)
{
    if (!n) return;
    for (int l = 0; l < 4; ++l)
        for (int b = 0; b < 2; ++b)
            for (int j = 0; j < 3; ++j) psg_mlp_destroy(n->sa[l].br[b].mlp[j]);
    for (int f = 0; f < 4; ++f)
        for (int j = 0; j < 3; ++j) psg_mlp_destroy(n->fp[f].mlp[j]);
    psg_mlp_destroy(n->conv1); psg_mlp_destroy(n->conv2);
    delete n;
}

extern "C" int psg_net_set_mlp_mode(psg_net *n, int mode)
{
    if (!n || mode < 0 || mode > 2) return PSG_EINVAL;
    n->mode = mode;
    return PSG_OK;
}

static PsgFpStream fp_stream_desc(psg_net *n, int f, int t, TView coarse);

extern "C" int psg_set_option(const char *name, int value)
{
    if (!name) return PSG_EINVAL;
    if (!strcmp(name, "nn_grid")) { psg_three_nn_grid_mode(value); return PSG_OK; }
    if (!strcmp(name, "fps_cluster")) { psg_fps_use_cluster(value); return PSG_OK; }
    if (!strcmp(name, "sa_compact")) { g_sa_compact = value != 0; return PSG_OK; }
    if (!strcmp(name, "x3_fused")) { g_x3_fused = value; return PSG_OK; }
    if (!strcmp(name, "stream_stages")) { psg_stream_tune(value, 0, 0); return PSG_OK; }
    if (!strcmp(name, "stream_stage_bytes")) { psg_stream_tune(0, value, 0); return PSG_OK; }
    if (!strcmp(name, "stream_rings")) { psg_stream_tune(0, 0, value); return PSG_OK; }
    return PSG_EINVAL;
}

extern "C" int psg_debug_trace(int64_t *buf, int nlaunches)
{
    psg_tile_set_trace(reinterpret_cast<long long *>(buf), buf ? nlaunches : 0);
    return PSG_OK;
}

extern "C" int psg_net_set_xyz_grad(psg_net *n, int on)
{
    if (!n) return PSG_EINVAL;
    n->xyz_grad = on != 0;
    return PSG_OK;
}

// carve (or, with base == null, only size) the workspace
static size_t plan(psg_net *n, int B, int N, int T, char *base)
{
    Bump bp{base, 0};
    const long long P = (long long)T * B;
    n->npts[0] = N;
    for (int l = 0; l < 4; ++l) n->npts[l + 1] = n->sa[l].S;
    n->xyz0 = bp.take<float>((size_t)B * N * 3);
    n->starts = bp.take<int>((size_t)4 * P);
    n->fps_ws_bytes = 0;
    size_t csr_scratch = 0, scratch = 0;
    for (int l = 1; l <= 4; ++l) {
        const int S = n->npts[l], R = n->npts[l - 1];
        n->xyz[l] = bp.take<float>((size_t)P * S * 3);
        n->fps_idx[l] = bp.take<int>((size_t)P * S);
        size_t w = psg_fps_workspace_bytes((int)P, R);
        if (w > n->fps_ws_bytes) n->fps_ws_bytes = w;
        SaLevel &L = n->sa[l - 1];
        for (int b = 0; b < L.nbr; ++b) {
            Branch &Br = L.br[b];
            const long long M = (long long)S * Br.K;
            Br.ball = bp.take<int>((size_t)P * M);
            Br.csr_off = bp.take<int>((size_t)P * (R + 1));
            Br.csr_perm = bp.take<int>((size_t)P * M);
            size_t c = psg_csr_scratch_bytes(P, (int)M, R);
            if (c > csr_scratch) csr_scratch = c;
            const long long rows = (long long)B * M;
            Br.G = bp.tl(rows, Br.gpad);
            size_t wmax = Br.gpad;
            for (int j = 0; j < Br.nl; ++j) {
                Br.Y[j] = bp.tl(rows, Br.mlp[j]->npad);
                if ((size_t)Br.mlp[j]->npad > wmax) wmax = Br.mlp[j]->npad;
            }
            Br.arg = bp.take<unsigned char>((size_t)B * S * Br.mlp[Br.nl - 1]->npad);
            Br.fused = Br.nl == 3 && psg_sa_fusable(Br.K, Br.gpad, Br.mlp[0]->npad, Br.mlp[1]->npad, Br.mlp[2]->npad);
            Br.streamed = !Br.fused && Br.nl == 3 &&
                          psg_sa_streamable(Br.K, Br.gpad, Br.mlp[0]->npad, Br.mlp[1]->npad, Br.mlp[2]->npad);
            Br.m0 = Br.m1 = nullptr;
            if (Br.fused || Br.streamed) {
                Br.m0 = bp.take<unsigned>(psg_sa_mask_words(rows, Br.mlp[0]->npad));
                Br.m1 = bp.take<unsigned>(psg_sa_mask_words(rows, Br.mlp[1]->npad));
            }
            Br.compactable = Br.fused && psg_sa_compactable(Br.K, Br.gpad, Br.mlp[0]->npad, Br.mlp[1]->npad, Br.mlp[2]->npad);
            memset(&Br.cp, 0, sizeof(Br.cp));
            if (Br.compactable) {
                char *cws = bp.take<char>(psg_sa_compact_bytes(P, T, S, Br.K));
                if (cws) Br.cp = psg_sa_compact_carve(cws, P, T, S, Br.K);
                Br.cp.cap = (long long)B * S * Br.K;
            }
            size_t s = (size_t)round_up_ll(rows, 128) * wmax;
            if (s > scratch) scratch = s;
        }
    }
    for (int f = 0; f < 4; ++f) {
        FpLevel &F = n->fp[f];
        const int Nf = n->npts[f], Nc = n->npts[f + 1];
        F.nn_idx = bp.take<int>((size_t)P * Nf * 3);
        F.nn_w = bp.take<float>((size_t)P * Nf * 3);
        F.csr_off = bp.take<int>((size_t)P * (Nc + 1));
        F.csr_perm = bp.take<int>((size_t)P * Nf * 3);
        size_t c = psg_csr_scratch_bytes(P, Nf * 3, Nc);
        if (c > csr_scratch) csr_scratch = c;
        const long long rows = (long long)B * Nf;
        F.I = bp.tl(rows, F.C2);
        size_t wmax = F.C1 + F.C2;
        for (int j = 0; j < F.nl; ++j) {
            F.Y[j] = bp.tl(rows, F.mlp[j]->npad);
            if ((size_t)F.mlp[j]->npad > wmax) wmax = F.mlp[j]->npad;
        }
        if (f == 0 && (size_t)n->conv1->npad > wmax) wmax = n->conv1->npad;
        F.Yrm = f > 0 ? bp.take<float>((size_t)round_up_ll(rows, 128) * F.mlp[F.nl - 1]->npad) : nullptr;
        F.streamed = false;
        for (int j = 0; j < 3; ++j) F.m[j] = nullptr;
        if (f > 0) {
            PsgFpStream q = fp_stream_desc(n, f, 0, TView{nullptr, 0, 0});
            F.streamed = psg_fp_streamable(q, true) && psg_fp_streamable(q, false) && (rows + 127) / 128 >= kFpMinTiles;
            if (F.streamed)
                for (int j = 0; j + 1 < F.nl; ++j) F.m[j] = bp.take<unsigned>(psg_sa_mask_words(rows, F.mlp[j]->npad));
        }
        size_t s = (size_t)round_up_ll(rows, 128) * wmax;
        if (s > scratch) scratch = s;
    }
    for (int l = 0; l <= 4; ++l) {
        n->feats[l] = bp.tl((long long)B * n->npts[l], n->wfeat[l]);
        n->dfeat[l] = bp.tl((long long)B * n->npts[l], n->wfeat[l]);
        size_t s = (size_t)round_up_ll((long long)B * n->npts[l], 128) * n->wfeat[l];
        if (s > scratch) scratch = s;
    }
    for (int l = 0; l <= 4; ++l) n->dxyz[l] = bp.take<float>((size_t)B * n->npts[l] * 3);
    n->xyz_tmp = bp.take<float>((size_t)B * N * 9);
    n->H = bp.tl((long long)B * N, n->conv1->npad);
    n->Z = bp.tl((long long)B * N, n->conv2->npad);
    n->dZ = bp.tl((long long)B * N, n->conv2->npad);
    n->scratch_floats = scratch;
    n->S[0] = bp.take<float>(scratch);
    n->S[1] = bp.take<float>(scratch);
    n->Srm = bp.take<float>(scratch);
    n->fps_ws = bp.take<char>(n->fps_ws_bytes ? n->fps_ws_bytes : 16);
    n->csr_ws = bp.take<char>(csr_scratch);
    n->grid_ws = N >= 2048 ? (void *)bp.take<char>(psg_ballgrid_workspace_bytes(B, N)) : nullptr;
    n->grid_valid = false;
    return bp.off + 1024;
}

extern "C" size_t psg_net_workspace(const psg_net *net, int B, int N, int T)
{
    if (!net || B <= 0 || N < 3 || T <= 0) return 0;
    psg_net tmp = *net;
    return plan(&tmp, B, N, T, nullptr);
}

extern "C" int psg_net_bind(psg_net *n, int B, int N, int T, void *ws, size_t ws_bytes)
{
    if (!n || !ws || B <= 0 || N < 3 || T <= 0) return PSG_EINVAL;
    if (((uintptr_t)ws & 1023) != 0) return PSG_EINVAL;
    for (int l = 0; l < 4; ++l)
        if (n->sa[l].S > (l == 0 ? N : n->sa[l - 1].S)) return PSG_EINVAL;
    psg_net tmp = *n;
    size_t need = plan(&tmp, B, N, T, nullptr);
    if (ws_bytes < need) return PSG_EWORKSPACE;
    plan(n, B, N, T, (char *)ws);
    n->B = B; n->N = N; n->T = T; n->bound = true; n->last_t = -1;
    return PSG_OK;
}

#define PSG_TRY(expr)                     \
    do {                                  \
        int rc__ = (expr);                \
        if (rc__ != PSG_OK) return rc__;  \
    } while (0)

extern "C" int psg_net_set_input(psg_net *n, const float *x, int64_t sb, int64_t sc, int64_t sn, psg_stream_t stream)
{
    if (!n || !n->bound || !x) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    PSG_RUN(PF_PACK, psg_pack_cf(x, sb, sc, sn, n->B, n->in_channels, n->N, TView{n->feats[0], n->wfeat[0] / 4, 0},
                                 n->wfeat[0], n->xyz0, st));
    n->grid_valid = false;
    return PSG_OK;
}

extern "C" int psg_net_copy_input(psg_net *n, const psg_net *src, psg_stream_t stream)
{
    if (!n || !src || !n->bound || !src->bound || n->B != src->B || n->N != src->N || n->wfeat[0] != src->wfeat[0]) return PSG_EINVAL;
    if (n == src) return PSG_OK;
    if (cudaMemcpyAsync(n->feats[0], src->feats[0], tl_bytes((long long)n->B * n->N, n->wfeat[0]), cudaMemcpyDeviceToDevice,
                        (cudaStream_t)stream) != cudaSuccess) return PSG_ECUDA;
    return PSG_OK;
}

// coordinates of level l for forward t
static inline const float *lvl_xyz(const psg_net *n, int l, int t)
{
    return l == 0 ? n->xyz0 : n->xyz[l] + (size_t)t * n->B * n->npts[l] * 3;
}

extern "C" int psg_net_geometry(psg_net *n, const int32_t *starts, int T, psg_stream_t stream)
{
    if (!n || !n->bound || !starts || T <= 0 || T > n->T) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = n->B;
    const int P = T * B;
    // starts arrive as [4][T][B] for this call's T (device memory)
    for (int l = 1; l <= 4; ++l) {
        const int R = n->npts[l - 1], S = n->npts[l];
        const float *cloud = l == 1 ? n->xyz0 : n->xyz[l - 1];
        const int nclouds = l == 1 ? B : P;
        const long long stride = (long long)R * 3;
        PSG_RUN(PF_FPS, psg_fps_launch(cloud, stride, nclouds, P, R, S, starts + (size_t)(l - 1) * P, n->fps_idx[l], n->xyz[l],
                               n->fps_ws, n->fps_ws_bytes, st));
        SaLevel &L = n->sa[l - 1];
        // MSG: the two radii of a level share one scan of the cloud (pointnet_util.py:246-248)
        int ns[2] = {L.br[0].K, L.nbr > 1 ? L.br[1].K : 0};
        if (l == 1 && n->grid_ws) {
            // level-0 clouds are shared by all T forwards: bin them once per input, query through the grid
            if (!n->grid_valid) {
                const double rmax = L.nbr > 1 && L.radius[1] > L.radius[0] ? L.radius[1] : L.radius[0];
                PSG_RUN(PF_BALL, psg_ballgrid_build(cloud, stride, nclouds, R, rmax, n->grid_ws, st));
                n->grid_valid = true;
            }
            PSG_RUN(PF_BALL, psg_ballgrid_query(n->grid_ws, cloud, stride, nclouds, P, R, n->xyz[l], S, L.nbr, L.radius, ns,
                                                L.br[0].ball, L.nbr > 1 ? L.br[1].ball : nullptr, st));
        } else
        PSG_RUN(PF_BALL, psg_ball_query_launch(cloud, stride, nclouds, P, R, n->xyz[l], S, L.nbr, L.radius, ns, L.br[0].ball,
                                      L.nbr > 1 ? L.br[1].ball : nullptr, st));
        for (int b = 0; b < L.nbr; ++b) {
            PSG_RUN(PF_CSR, psg_csr_build(L.br[b].ball, P, S * L.br[b].K, R, L.br[b].K, L.br[b].csr_off, L.br[b].csr_perm, n->csr_ws, st));
            // compacted rows of the fused branches (skipped when the coordinates move: the geometric-gradient kernels
            // read the padded [S][K] layout)
            if (L.br[b].compactable && g_sa_compact && n->mode >= 1 && !n->xyz_grad)
                PSG_RUN(PF_CSR, psg_sa_compact_build(L.br[b].ball, L.br[b].csr_perm, T, B, S, L.br[b].K, L.br[b].cp, st));
        }
        n->compact_valid = g_sa_compact && n->mode >= 1 && !n->xyz_grad;
    }
    for (int f = 0; f < 4; ++f) {
        FpLevel &F = n->fp[f];
        const int Nf = n->npts[f], Nc = n->npts[f + 1];
        const float *fine = f == 0 ? n->xyz0 : n->xyz[f];
        PSG_RUN(PF_NN3, psg_three_nn_launch(fine, (long long)Nf * 3, f == 0 ? B : P, P, Nf, n->xyz[f + 1], Nc, F.nn_idx, F.nn_w,
                                    nullptr, st));
        PSG_RUN(PF_CSR, psg_csr_build(F.nn_idx, P, Nf * 3, Nc, 0, F.csr_off, F.csr_perm, n->csr_ws, st));
    }
    return PSG_OK;
}

extern "C" int psg_net_read_geometry(const psg_net *n, int what, int level, int branch, int t, void *dst, size_t dst_bytes,
                                     psg_stream_t stream)
{
    if (!n || !n->bound || !dst || t < 0 || t >= n->T) return PSG_EINVAL;
    const size_t B = n->B;
    const void *src = nullptr;
    size_t bytes = 0;
    if (what == 0 || what == 4) {
        if (level < 1 || level > 4) return PSG_EINVAL;
        const size_t S = n->npts[level];
        if (what == 0) { src = n->fps_idx[level] + (size_t)t * B * S; bytes = B * S * sizeof(int); }
        else { src = n->xyz[level] + (size_t)t * B * S * 3; bytes = B * S * 3 * sizeof(float); }
    } else if (what == 1) {
        if (level < 1 || level > 4 || branch < 0 || branch >= n->sa[level - 1].nbr) return PSG_EINVAL;
        const Branch &Br = n->sa[level - 1].br[branch];
        const size_t M = (size_t)n->npts[level] * Br.K;
        src = Br.ball + (size_t)t * B * M; bytes = B * M * sizeof(int);
    } else if (what == 2 || what == 3) {
        if (level < 0 || level > 3) return PSG_EINVAL;
        const size_t Nf = n->npts[level];
        if (what == 2) src = n->fp[level].nn_idx + (size_t)t * B * Nf * 3;
        else src = n->fp[level].nn_w + (size_t)t * B * Nf * 3;
        bytes = B * Nf * 3 * 4;
    } else
        return PSG_EINVAL;
    if (dst_bytes < bytes) return PSG_EWORKSPACE;
    if (cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream) != cudaSuccess) return PSG_ECUDA;
    return PSG_OK;
}

static inline TView tv(float *p, int width, int col0 = 0) { return TView{p, width / 4, col0 / 4}; }

// fp1 + head as one forward + backward kernel: the TF32 mode always, the 3xTF32 mode with x3_fused bit 1
static inline bool head_fused_now(const psg_net *n)
{
    return n->head_fused && (n->mode == 1 || (n->mode == 2 && (g_x3_fused & 2)));
}

// does the branch run as one kernel per direction in the network's current mode?
static inline bool branch_fused_now(const psg_net *n, const Branch &Br)
{
    if (n->mode == 1) return Br.fused || Br.streamed;
    if (n->mode == 2)
        return (g_x3_fused & 1) && Br.fused && Br.compactable && n->compact_valid && !n->xyz_grad &&
               psg_sa_fusable_x3(Br.K, Br.gpad, Br.mlp[0]->npad, Br.mlp[1]->npad, Br.mlp[2]->npad);
    return false;
}

static PsgSaFused sa_fused_desc(psg_net *n, int l, int b, int t)
{
    SaLevel &L = n->sa[l - 1];
    Branch &Br = L.br[b];
    const int B = n->B, S = L.S, R = n->npts[l - 1];
    PsgSaFused f;
    f.K = Br.K;
    f.feats = tv(n->feats[l - 1], n->wfeat[l - 1]); f.D = n->cfeat[l - 1];
    f.xyz = lvl_xyz(n, l - 1, t); f.cloud_stride = (long long)R * 3; f.nclouds = B; f.Nsrc = R;
    f.new_xyz = lvl_xyz(n, l, t); f.idx = Br.ball + (size_t)t * B * S * Br.K;
    f.rows = (long long)B * S * Br.K; f.S = S;
    f.gpad = Br.gpad;
    const bool x3 = n->mode == 2;
    for (int j = 0; j < 3; ++j) {
        f.n[j] = Br.mlp[j]->npad;
        f.wf[j] = w_fwd(Br.mlp[j], x3 ? 2 : 1); f.nwf[j] = Br.mlp[j]->nwf; f.bias[j] = Br.mlp[j]->bias;      // (fused = tcgen05 only)
        f.wb[j] = w_bwd(Br.mlp[j], x3 ? 2 : 1); f.nwb[j] = Br.mlp[j]->nwb;
        f.wf_lo[j] = x3 ? Br.mlp[j]->wf_lo : nullptr;     // mode 2: 3xTF32 inside the fused kernels (sa_fused.cu)
        f.wb_lo[j] = x3 ? Br.mlp[j]->wb_lo : nullptr;
    }
    f.m0 = Br.m0; f.m1 = Br.m1;
    f.out = tv(n->feats[l], n->wfeat[l], Br.col0); f.arg = Br.arg;
    f.crow_src = f.crow_g = f.ntiles_dev = nullptr;
    if (Br.compactable && n->compact_valid) {
        f.crow_src = Br.cp.crow_src + (size_t)t * Br.cp.cap;
        f.crow_g = Br.cp.crow_g + (size_t)t * Br.cp.cap;
        f.ntiles_dev = Br.cp.ctiles + t;
    }
    return f;
}

// feature-propagation level f >= 1 (fine level f, coarse level f + 1) as a tile program
static PsgFpStream fp_stream_desc(psg_net *n, int f, int t, TView coarse)
{
    FpLevel &F = n->fp[f];
    const int B = n->B, Nf = n->npts[f], Nc = n->npts[f + 1];
    PsgFpStream q;
    memset(&q, 0, sizeof(q));
    q.skip = tv(n->feats[f], n->wfeat[f]); q.C1 = F.C1;
    q.coarse = coarse; q.C2 = F.C2; q.S = Nc; q.Nf = Nf; q.rows = (long long)B * Nf;
    q.nn_idx = F.nn_idx + (size_t)t * B * Nf * 3; q.nn_w = F.nn_w + (size_t)t * B * Nf * 3;
    q.nl = F.nl;
    for (int j = 0; j < F.nl; ++j) {
        const psg_mlp *m = F.mlp[j];
        q.n[j] = m->npad; q.wf[j] = w_fwd(m, 1); q.nwf[j] = m->nwf; q.bias[j] = m->bias; q.wb[j] = w_bwd(m, 1); q.nwb[j] = m->nwb;
        q.m[j] = F.m[j];
    }
    q.y_last = tv(F.Y[F.nl - 1], F.mlp[F.nl - 1]->npad);
    q.y_last_rm = F.Yrm;
    // the coarser level's mirror exists only if that level ran as a tile program too
    q.coarse_rm = (f < 3 && n->fp[f + 1].streamed && n->mode == 1) ? n->fp[f + 1].Yrm : nullptr;
    return q;
}

// fp1 (+ conv1 as one more hidden layer) + conv2 head, interpolating from `coarse` (fp2's output)
static PsgChain head_chain_desc(psg_net *n, int t, TView coarse)
{
    FpLevel &F = n->fp[0];
    const int B = n->B, Nf = n->npts[0], Nc = n->npts[1];
    PsgChain c;
    memset(&c, 0, sizeof(c));
    c.src = coarse; c.S = Nc; c.Nf = Nf; c.kin = F.C2; c.rows = (long long)B * Nf;
    c.nn_idx = F.nn_idx + (size_t)t * B * Nf * 3; c.nn_w = F.nn_w + (size_t)t * B * Nf * 3;
    c.nlayers = F.nl + 1;
    const int wm = n->mode == 2 ? 2 : 1;           // mode 2: hi parts here, residuals below (3xTF32 inside the tile program)
    for (int j = 0; j <= F.nl; ++j) {
        const psg_mlp *m = j < F.nl ? F.mlp[j] : n->conv1;
        c.n[j] = m->npad; c.wf[j] = w_fwd(m, wm); c.nwf[j] = m->nwf; c.bias[j] = m->bias; c.wb[j] = w_bwd(m, wm); c.nwb[j] = m->nwb;
        if (wm == 2) { c.wf_lo[j] = m->wf_lo; c.wb_lo[j] = m->wb_lo; }
    }
    c.head_wf = w_fwd(n->conv2, wm); c.head_nwf = n->conv2->nwf; c.head_bias = n->conv2->bias;
    c.head_wb = w_bwd(n->conv2, wm); c.head_nwb = n->conv2->nwb;
    if (wm == 2) { c.head_wf_lo = n->conv2->wf_lo; c.head_wb_lo = n->conv2->wb_lo; }
    c.ncls = n->ncls; c.target = -1;
    c.src_rm = (n->fp[1].streamed && n->mode == 1) ? n->fp[1].Yrm : nullptr;
    return c;
}

extern "C" int psg_net_forward(psg_net *n, int t, float *logp, float *l4_points, psg_stream_t stream)
{
    if (!n || !n->bound || t < 0 || t >= n->T) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = n->B, mode = n->mode;
    const TView none{nullptr, 0, 0};
    for (int l = 1; l <= 4; ++l) {
        SaLevel &L = n->sa[l - 1];
        const int S = L.S, R = n->npts[l - 1], D = n->cfeat[l - 1];
        for (int b = 0; b < L.nbr; ++b) {
            Branch &Br = L.br[b];
            const long long rows = (long long)B * S * Br.K;
            if (branch_fused_now(n, Br)) {
                PsgSaFused f = sa_fused_desc(n, l, b, t);
                PSG_RUN(PF_SA_FWD, Br.fused ? psg_sa_fused_fwd(f, st) : psg_sa_stream_fwd(f, st));
                continue;
            }
            PSG_RUN(PF_GROUP, psg_group(tv(n->feats[l - 1], n->wfeat[l - 1]), D, lvl_xyz(n, l - 1, t), (long long)R * 3, B, R,
                              lvl_xyz(n, l, t), Br.ball + (size_t)t * B * S * Br.K, B, S, Br.K, tv(Br.G, Br.gpad), Br.gpad,
                              st));
            TView cur = tv(Br.G, Br.gpad);
            int kw = Br.gpad;
            for (int j = 0; j < Br.nl; ++j) {
                TView out = tv(Br.Y[j], Br.mlp[j]->npad);
                PSG_RUN(PF_GEMM_FWD, mlp_fwd(Br.mlp[j], cur, kw / 4, none, 0, rows, out, 1, mode, st));
                cur = out; kw = Br.mlp[j]->npad;
            }
            PSG_RUN(PF_MAXPOOL, psg_maxpool(cur, (long long)B * S, Br.K, kw, tv(n->feats[l], n->wfeat[l], Br.col0), Br.arg, st));
        }
    }
    // feature propagation, coarse to fine
    float *up = n->feats[4];
    int upw = n->wfeat[4];
    const bool fuse_head = head_fused_now(n);
    n->z_valid = false;
    n->loss.set = false;
    for (int f = 3; f >= 0; --f) {
        FpLevel &F = n->fp[f];
        const int Nf = n->npts[f], Nc = n->npts[f + 1];
        const long long rows = (long long)B * Nf;
        if (f == 0 && fuse_head) {
            // fp1 + head as one kernel; when nobody asked for the log-probabilities the whole chain is
            // deferred to psg_net_backward, which runs it forward AND backward in one pass
            if (logp) {
                PsgChain c = head_chain_desc(n, t, tv(up, upw));
                c.backward = 0; c.zout = tv(n->Z, n->conv2->npad);
                PSG_RUN(PF_HEAD_CHAIN, psg_chain_fused(c, st));
                n->z_valid = true;
            }
            break;
        }
        if (mode == 1 && F.streamed) {
            PsgFpStream q = fp_stream_desc(n, f, t, tv(up, upw));
            PSG_RUN(PF_FP_FWD, psg_fp_stream_fwd(q, st));
            up = F.Y[F.nl - 1]; upw = F.mlp[F.nl - 1]->npad;
            continue;
        }
        PSG_RUN(PF_INTERP, psg_interp(tv(up, upw), Nc, F.nn_idx + (size_t)t * B * Nf * 3, F.nn_w + (size_t)t * B * Nf * 3, B, Nf,
                           F.C2 / 4, tv(F.I, F.C2), st));
        TView a1 = F.C1 ? tv(n->feats[f], n->wfeat[f]) : tv(F.I, F.C2);
        TView a2 = F.C1 ? tv(F.I, F.C2) : none;
        int k1 = F.C1 ? F.C1 / 4 : F.C2 / 4, k2 = F.C1 ? F.C2 / 4 : 0;
        for (int j = 0; j < F.nl; ++j) {
            TView out = tv(F.Y[j], F.mlp[j]->npad);
            PSG_RUN(PF_GEMM_FWD, mlp_fwd(F.mlp[j], a1, k1, a2, k2, rows, out, 1, mode, st));
            a1 = out; k1 = F.mlp[j]->npad / 4; a2 = none; k2 = 0;
        }
        up = F.Y[F.nl - 1]; upw = F.mlp[F.nl - 1]->npad;
    }
    const long long rows0 = (long long)B * n->N;
    if (!fuse_head) {
        PSG_RUN(PF_GEMM_FWD, mlp_fwd(n->conv1, tv(up, upw), upw / 4, none, 0, rows0, tv(n->H, n->conv1->npad), 1, mode, st));
        PSG_RUN(PF_GEMM_FWD, mlp_fwd(n->conv2, tv(n->H, n->conv1->npad), n->conv1->npad / 4, none, 0, rows0,
                                     tv(n->Z, n->conv2->npad), 0, mode, st));
        n->z_valid = true;
    }
    if (logp) PSG_RUN(PF_HEAD, psg_head_logsoftmax(tv(n->Z, n->conv2->npad), rows0, n->ncls, logp, st));
    if (l4_points) PSG_RUN(PF_PACK, psg_unpack_cf(tv(n->feats[4], n->wfeat[4]), B, n->cfeat[4], n->npts[4], l4_points, 0, st));
    n->last_t = t;
    return PSG_OK;
}

static int set_loss(psg_net *n, int kind, const float *dlogp, const int32_t *labels, int target, float scale, float kappa,
                    float *loss_rows, unsigned char *hit, cudaStream_t st)
{
    if (kind == 0 && !dlogp) return PSG_EINVAL;
    if (kind != 0 && !labels && target < 0) return PSG_EINVAL;
    if (kind < 0 || kind > 2) return PSG_EINVAL;
    if (head_fused_now(n)) {
        // evaluated inside the fused fp1 + head kernel launched by psg_net_backward
        n->loss.kind = kind; n->loss.dlogp = dlogp; n->loss.labels = labels; n->loss.target = target;
        n->loss.scale = scale; n->loss.kappa = kappa; n->loss.loss_rows = loss_rows; n->loss.hit = hit; n->loss.set = true;
        return PSG_OK;
    }
    const long long rows = (long long)n->B * n->N;
    TView z = tv(n->Z, n->conv2->npad), dz = tv(n->dZ, n->conv2->npad);
    if (kind == 0) PSG_RUN(PF_LOSS, psg_dz_from_dlogp(z, dlogp, rows, n->ncls, dz, st));
    else if (kind == 1) PSG_RUN(PF_LOSS, psg_dz_ce(z, labels, target, rows, n->ncls, scale, dz, st));
    else PSG_RUN(PF_LOSS, psg_dz_cw(z, labels, target, rows, n->ncls, kappa, scale, dz, loss_rows, hit, st));
    return PSG_OK;
}

extern "C" int psg_net_loss_grad(psg_net *n, int kind, const float *dlogp, const int32_t *labels, int target, float scale,
                                 float kappa, float *loss_rows, psg_stream_t stream)
{
    if (!n || !n->bound || n->last_t < 0) return PSG_EINVAL;
    return set_loss(n, kind, dlogp, labels, target, scale, kappa, loss_rows, nullptr, (cudaStream_t)stream);
}

// Backward through a chain of folded layers.  `top` is the gradient w.r.t. the pre-activation of
// the last layer; Ys[j] the forward output of layer j.  Ping-pongs between the two scratch buffers,
// starting with the one `top` does not live in; returns the buffer index holding dIn.
static int chain_bwd(psg_net *n, psg_mlp *const *mlps, float *const *Ys, int nl, long long rows, TView top, int top_buf,
                     int *out_buf, cudaStream_t st, const TView *out2 = nullptr, int out2_cols = 0)
{
    TView cur = top;
    int dstb = top_buf == 0 ? 1 : 0;
    for (int j = nl - 1; j >= 0; --j) {
        TView dx = tv(n->S[dstb], mlps[j]->kpad);
        if (j > 0) {
            TView mk = tv(Ys[j - 1], mlps[j - 1]->npad);
            PSG_RUN(PF_GEMM_BWD, mlp_bwd(mlps[j], cur, rows, dx, &mk, n->mode, st));
        } else {
            PSG_RUN(PF_GEMM_BWD, mlp_bwd(mlps[j], cur, rows, dx, nullptr, n->mode, st, out2, out2_cols));
        }
        cur = dx;
        *out_buf = dstb;
        dstb ^= 1;
    }
    return PSG_OK;
}

extern "C" int psg_net_backward(psg_net *n, int t, float *grad_x, psg_stream_t stream)
{
    if (!n || !n->bound || t < 0 || t >= n->T || t != n->last_t) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = n->B;
    // the geometric-gradient kernels read the padded [S][K] gradient rows: the geometry must have been built with the
    // coordinate gradient already switched on (psg_net_set_xyz_grad before psg_net_geometry)
    if (n->xyz_grad && n->compact_valid) return PSG_EINVAL;
    if (n->xyz_grad)
        for (int l = 0; l <= 4; ++l)
            if (cudaMemsetAsync(n->dxyz[l], 0, (size_t)B * n->npts[l] * 3 * sizeof(float), st) != cudaSuccess) return PSG_ECUDA;
    // ---- head + feature propagation, fine to coarse ----
    TView top = tv(n->dZ, n->conv2->npad);
    int top_buf = -1;
    for (int f = 0; f <= 3; ++f) {
        FpLevel &F = n->fp[f];
        const int Nf = n->npts[f], Nc = n->npts[f + 1];
        const long long rows = (long long)B * Nf;
        psg_mlp *mlps[5]; float *Ys[5]; int nl = 0;
        for (int j = 0; j < F.nl; ++j) { mlps[nl] = F.mlp[j]; Ys[nl] = F.Y[j]; ++nl; }
        if (f == 0) { mlps[nl] = n->conv1; Ys[nl] = n->H; ++nl; mlps[nl] = n->conv2; Ys[nl] = n->Z; ++nl; }
        int cat_buf = 0;
        const float *rm_src = nullptr; int rm_stride = 0;      // row-major copy of d[interp] when a fused kernel produced it
        int skip_done = 0;                                      // leading columns of d[skip] the producing kernel already wrote into dfeat[f]
        if (f == 0 && head_fused_now(n)) {
            if (!n->loss.set) return PSG_EINVAL;
            FpLevel &C = n->fp[1];
            PsgChain c = head_chain_desc(n, t, tv(C.Y[C.nl - 1], C.mlp[C.nl - 1]->npad));
            c.backward = 1; c.loss_kind = n->loss.kind; c.target = n->loss.target; c.labels = n->loss.labels;
            c.scale = n->loss.scale; c.kappa = n->loss.kappa; c.dlogp = n->loss.dlogp;
            c.loss_rows = n->loss.loss_rows; c.hit = n->loss.hit;
            c.dI = tv(n->S[0], F.C2);
            c.dI_rm = n->Srm; c.rm_only = n->xyz_grad ? 0 : 1;
            rm_src = n->Srm; rm_stride = F.C2;
            PSG_RUN(PF_HEAD_CHAIN, psg_chain_fused(c, st));
        } else if (f > 0 && n->mode == 1 && F.streamed) {
            PsgFpStream q = fp_stream_desc(n, f, t, TView{nullptr, 0, 0});
            cat_buf = top_buf == 0 ? 1 : 0;
            // the skip part of the gradient goes straight into dfeat[f] as far as the tile program covers it
            PSG_RUN(PF_FP_BWD, psg_fp_stream_bwd(q, top, tv(n->S[cat_buf], F.C1 + F.C2), n->Srm, tv(n->dfeat[f], n->wfeat[f]), st));
            rm_src = n->Srm + F.C1; rm_stride = F.C1 + F.C2;
            skip_done = psg_fp_stream_skip_cols(q);
        } else if (f > 0 && n->mode >= 1 && F.C1) {
            TView dsk = tv(n->dfeat[f], n->wfeat[f]);
            PSG_TRY(chain_bwd(n, mlps, Ys, nl, rows, top, top_buf, &cat_buf, st, &dsk, F.C1));
            skip_done = F.C1;
        } else {
            PSG_TRY(chain_bwd(n, mlps, Ys, nl, rows, top, top_buf, &cat_buf, st));
        }
        const int catw = F.C1 + F.C2;
        if (F.C1 > skip_done)
            PSG_RUN(PF_COPY, psg_copy_cols(tv(n->S[cat_buf], catw, skip_done), tv(n->dfeat[f], n->wfeat[f], skip_done), rows,
                                           F.C1 - skip_done, 0, st));
        // interpolation backward: scatter the three weighted copies to the coarse level, in CSR order
        const size_t go = (size_t)t * B;
        if (n->xyz_grad) {
            // d cost / d coordinates through the inverse-distance weights (pointnet_util.py:301-308)
            float *coarse = f < 3 ? n->fp[f + 1].Y[n->fp[f + 1].nl - 1] : n->feats[4];
            const int cw2 = f < 3 ? n->fp[f + 1].mlp[n->fp[f + 1].nl - 1]->npad : n->wfeat[4];
            PSG_RUN(PF_SEGSUM, psg_fp_xyz_backward(tv(n->S[cat_buf], catw, F.C1), tv(coarse, cw2), F.C2, lvl_xyz(n, f, t),
                                                   (long long)Nf * 3, B, lvl_xyz(n, f + 1, t), Nc, F.nn_idx + go * Nf * 3,
                                                   F.csr_off + go * (Nc + 1), F.csr_perm + go * Nf * 3, B, Nf, n->dxyz[f],
                                                   n->dxyz[f + 1], n->xyz_tmp, st));
        }
        if (f < 3) {
            FpLevel &C = n->fp[f + 1];
            const int cw = C.mlp[C.nl - 1]->npad;
            const int dst_buf = cat_buf ^ 1;
            TView dst = tv(n->S[dst_buf], cw);
            TView mk = tv(C.Y[C.nl - 1], cw);
            PSG_RUN(PF_SEGSUM, psg_segsum(tv(n->S[cat_buf], catw, F.C1), Nf, 3, F.nn_w + go * Nf * 3, F.csr_off + go * (Nc + 1),
                                          F.csr_perm + go * Nf * 3, Nf * 3, Nc, B, F.C2, dst, 0, &mk, rm_src, rm_stride, st));
            top = dst; top_buf = dst_buf;
        } else {
            PSG_RUN(PF_SEGSUM, psg_segsum(tv(n->S[cat_buf], catw, F.C1), Nf, 3, F.nn_w + go * Nf * 3, F.csr_off + go * (Nc + 1),
                                          F.csr_perm + go * Nf * 3, Nf * 3, Nc, B, F.C2, tv(n->dfeat[4], n->wfeat[4]), 0, nullptr,
                                          rm_src, rm_stride, st));
        }
    }
    // ---- set abstraction, coarse to fine ----
    for (int l = 4; l >= 1; --l) {
        SaLevel &L = n->sa[l - 1];
        const int S = L.S, R = n->npts[l - 1], D = n->cfeat[l - 1];
        for (int b = 0; b < L.nbr; ++b) {
            Branch &Br = L.br[b];
            const long long rows = (long long)B * S * Br.K;
            const int cw = Br.mlp[Br.nl - 1]->npad;
            if (branch_fused_now(n, Br)) {
                PsgSaFused f = sa_fused_desc(n, l, b, t);
                // feature columns only, unless the coordinate gradient is wanted too
                const int gcols = n->xyz_grad ? Br.gpad : round_up(D, 16);
                TView dl = tv(n->dfeat[l], n->wfeat[l], Br.col0), dg = tv(n->S[0], Br.gpad);
                const int rmo = n->xyz_grad ? 0 : 1;
                PSG_RUN(PF_SA_BWD, Br.fused ? psg_sa_fused_bwd(f, dl, dg, gcols, n->Srm, rmo, st) : psg_sa_stream_bwd(f, dl, dg, gcols, n->Srm, rmo, st));
                const size_t go = (size_t)t * B;
                const int M = S * Br.K;
                if (f.crow_src)      // compacted gradient rows: the permutation addresses them relative to the forward
                    PSG_RUN(PF_SEGSUM, psg_segsum(tv(n->S[0], Br.gpad), 0, 1, nullptr, Br.csr_off + go * (R + 1), Br.cp.cperm + go * M, M, R,
                                       B, D, tv(n->dfeat[l - 1], n->wfeat[l - 1]), (l > 1 || b > 0) ? 1 : 0, nullptr, n->Srm, Br.gpad, st));
                else
                PSG_RUN(PF_SEGSUM, psg_segsum(tv(n->S[0], Br.gpad), M, 1, nullptr, Br.csr_off + go * (R + 1), Br.csr_perm + go * M, M, R,
                                   B, D, tv(n->dfeat[l - 1], n->wfeat[l - 1]), (l > 1 || b > 0) ? 1 : 0, nullptr, n->Srm, Br.gpad, st));
                if (n->xyz_grad)
                    PSG_RUN(PF_SEGSUM, psg_sa_xyz_backward(tv(n->S[0], Br.gpad), D, Br.K, S, B, Br.csr_off + go * (R + 1),
                                                           Br.csr_perm + go * M, R, n->dxyz[l - 1], n->dxyz[l], st));
                continue;
            }
            TView dy = tv(n->S[0], cw);
            PSG_RUN(PF_MAXPOOL_BWD, psg_maxpool_bwd(tv(n->dfeat[l], n->wfeat[l], Br.col0), tv(n->feats[l], n->wfeat[l], Br.col0), Br.arg,
                                    (long long)B * S, Br.K, cw, dy, st));
            int gbuf = 0;
            PSG_TRY(chain_bwd(n, Br.mlp, Br.Y, Br.nl, rows, dy, 0, &gbuf, st));
            const size_t go = (size_t)t * B;
            const int M = S * Br.K;
            PSG_RUN(PF_SEGSUM, psg_segsum(tv(n->S[gbuf], Br.gpad), M, 1, nullptr, Br.csr_off + go * (R + 1), Br.csr_perm + go * M, M, R,
                               B, D, tv(n->dfeat[l - 1], n->wfeat[l - 1]), (l > 1 || b > 0) ? 1 : 0, nullptr, nullptr, 0, st));
            if (n->xyz_grad)
                PSG_RUN(PF_SEGSUM, psg_sa_xyz_backward(tv(n->S[gbuf], Br.gpad), D, Br.K, S, B, Br.csr_off + go * (R + 1),
                                                       Br.csr_perm + go * M, R, n->dxyz[l - 1], n->dxyz[l], st));
        }
        // xyz_l = xyz_{l-1}[fps_idx]: everything that reached the centroids' coordinates flows to their source points
        if (n->xyz_grad)
            PSG_RUN(PF_SEGSUM, psg_fps_xyz_backward(n->dxyz[l], n->fps_idx[l] + (size_t)t * B * S, S, R, B, n->dxyz[l - 1], st));
    }
    if (n->xyz_grad) PSG_RUN(PF_SEGSUM, psg_add_xyz_to_feat(n->dxyz[0], (long long)B * n->N, tv(n->dfeat[0], n->wfeat[0]), st));
    if (grad_x) PSG_RUN(PF_PACK, psg_unpack_cf(tv(n->dfeat[0], n->wfeat[0]), B, n->in_channels, n->N, grad_x, 0, st));
    return PSG_OK;
}

extern "C" int psg_net_pgd_update(psg_net *n, float *adv, const float *ori, const uint8_t *mask, int c0, int nc,
                                  float alpha_signed, float eps, float lo, float hi, psg_stream_t stream)
{
    if (!n || !n->bound || !adv || !ori || c0 < 0 || nc <= 0 || c0 + nc > n->in_channels) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    PSG_RUN(PF_PGD, psg_pgd_update(adv, ori, tv(n->dfeat[0], n->wfeat[0]), tv(n->feats[0], n->wfeat[0]), mask, n->B,
                                   n->in_channels, n->N, c0, nc, alpha_signed, eps, lo, hi, st));
    return PSG_OK;
}

// torchattacks PGDL2's step and projection on the same field (elementwise.cu, pgd_l2_update_kernel): the norms are taken
// per block over its moving points, so eps is an L2 radius in colour space
extern "C" int psg_net_pgd_update_l2(psg_net *n, float *adv, const float *ori, const uint8_t *mask, int c0, int nc,
                                     float alpha_signed, float eps, float lo, float hi, psg_stream_t stream)
{
    if (!n || !n->bound || !adv || !ori || c0 < 0 || nc <= 0 || c0 + nc > n->in_channels) return PSG_EINVAL;
    if (!std::isfinite(alpha_signed) || !std::isfinite(eps) || eps < 0.f) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    PSG_RUN(PF_PGD, psg_pgd_l2_update(adv, ori, tv(n->dfeat[0], n->wfeat[0]), tv(n->feats[0], n->wfeat[0]), mask, n->B,
                                      n->in_channels, n->N, c0, nc, alpha_signed, eps, lo, hi, st));
    return PSG_OK;
}

// The NB / tar-NB loop body shared by both norms: forward, cross-entropy gradient, backward, update on colours 3:6.
static int nb_loop(psg_net *n, bool l2, float *adv, const float *ori, const uint8_t *mask, const int32_t *labels, int target,
                   int iters, int t0, float alpha, float eps, float scale, psg_stream_t stream)
{
    if (!n || !n->bound || iters < 0 || t0 < 0 || t0 + iters > n->T) return PSG_EINVAL;
    if (l2 && (!std::isfinite(alpha) || !std::isfinite(eps) || eps < 0.f)) return PSG_EINVAL;
    // non-targeted: ascent on the true-label cost (nontarget.py:37); targeted: descent on the
    // target-label cost (target.py:41)
    const float a = target >= 0 ? -alpha : alpha;
    for (int i = 0; i < iters; ++i) {
        PSG_TRY(psg_net_forward(n, t0 + i, nullptr, nullptr, stream));
        PSG_TRY(psg_net_loss_grad(n, 1, nullptr, labels, target, scale, 0.f, nullptr, stream));
        PSG_TRY(psg_net_backward(n, t0 + i, nullptr, stream));
        PSG_TRY(l2 ? psg_net_pgd_update_l2(n, adv, ori, mask, 3, 3, a, eps, 0.f, 1.f, stream)
                   : psg_net_pgd_update(n, adv, ori, mask, 3, 3, a, eps, 0.f, 1.f, stream));
    }
    return PSG_OK;
}

extern "C" int psg_nb_attack(psg_net *n, float *adv, const float *ori, const uint8_t *mask, const int32_t *labels,
                             int target, int iters, int t0, float alpha, float eps, float scale, psg_stream_t stream)
{
    return nb_loop(n, false, adv, ori, mask, labels, target, iters, t0, alpha, eps, scale, stream);
}

extern "C" int psg_nb_attack_l2(psg_net *n, float *adv, const float *ori, const uint8_t *mask, const int32_t *labels,
                                int target, int iters, int t0, float alpha, float eps, float scale, psg_stream_t stream)
{
    return nb_loop(n, true, adv, ori, mask, labels, target, iters, t0, alpha, eps, scale, stream);
}

// ------------------------------------------------------------------------------------------------
// norm-unbounded attacks (nontarget.py:52-106, target.py:62-133): one step = one launch sequence
// ------------------------------------------------------------------------------------------------
namespace {
struct NuScratch { float *f_rows, *l2_rows, *smooth_rows, *smooth_grad; unsigned char *hit; };
inline NuScratch nu_carve(float *s, int B, int N)
{
    const size_t bn = (size_t)B * N;
    NuScratch r;
    r.f_rows = s; r.l2_rows = s + bn; r.smooth_rows = s + 2 * bn; r.smooth_grad = r.smooth_rows + N;
    r.hit = reinterpret_cast<unsigned char *>(r.smooth_grad + 3 * (size_t)N);
    return r;
}
}  // namespace

extern "C" size_t psg_nu_scratch_floats(int B, int N)
{
    if (B <= 0 || N <= 0) return 0;
    const size_t bn = (size_t)B * N;
    return 2 * bn + 4 * (size_t)N + (bn + 3) / 4 + 16;
}

static int nu_field(const psg_net *n, const psg_nu_buffers *b, PsgNuField *f)
{
    if (b->field_nc == 0) {                       // the reference's field: colours 3:6 in [0, 1]
        f->c0 = 3; f->nc = 3;
        for (int j = 0; j < 8; ++j) { f->lo[j] = 0.f; f->hi[j] = 1.f; }
        return PSG_OK;
    }
    if (b->field_c0 < 0 || b->field_nc < 1 || b->field_nc > 8 || b->field_c0 + b->field_nc > n->in_channels) return PSG_EINVAL;
    f->c0 = b->field_c0; f->nc = b->field_nc;
    for (int j = 0; j < 8; ++j) {
        f->lo[j] = j < f->nc ? b->box_lo[j] : 0.f;
        f->hi[j] = j < f->nc ? b->box_hi[j] : 1.f;
        if (j < f->nc && !(f->hi[j] > f->lo[j])) return PSG_EINVAL;
    }
    return PSG_OK;
}

extern "C" int psg_nu_init(psg_net *n, const psg_nu_buffers *b, psg_stream_t stream)
{
    if (!n || !n->bound || !b || !b->w || !b->adam_m || !b->adam_v || !b->images || !b->status) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    PsgNuField fld;
    PSG_TRY(nu_field(n, b, &fld));
    if (cudaMemsetAsync(b->status, 0, 4 * sizeof(int32_t), st) != cudaSuccess) return PSG_ECUDA;
    PSG_RUN(PF_PGD, psg_nu_init_k(b->images, n->B, n->in_channels, n->N, fld, b->w, b->adam_m, b->adam_v, st));
    return PSG_OK;
}

extern "C" int psg_nu_step(psg_net *n, const psg_nu_buffers *b, int t, int step, int target, int neighbour, float c,
                           float kappa, float targeted_sign, float step_size, float bc2_sqrt, int reset_adam,
                           double acc_denom, double thr, int exit_above, int count_masked_only, const int32_t *starts,
                           psg_stream_t stream)
{
    if (!n || !n->bound || !b || !b->w || !b->adv || !b->base || !b->images || !b->labels || !b->cost || !b->status ||
        !b->scratch || step < 0 || acc_denom <= 0.0)
        return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = n->B, N = n->N, C = n->in_channels;
    const long long rows = (long long)B * N;
    NuScratch s = nu_carve(b->scratch, B, N);
    TView f0 = tv(n->feats[0], n->wfeat[0]), g0 = tv(n->dfeat[0], n->wfeat[0]);
    PsgNuField fld;
    PSG_TRY(nu_field(n, b, &fld));
    PSG_RUN(PF_PGD, psg_nu_build_adv_k(b->w, b->base, b->images, b->mask, B, C, N, fld, f0, b->adv, s.l2_rows, b->status, st));
    if (fld.c0 < 3) {
        // the coordinates moved: refresh xyz from the step's image and rebuild the geometry of slot t
        if (!starts || t != 0) return PSG_EINVAL;
        PSG_TRY(psg_net_set_input(n, b->adv, (int64_t)C * N, N, 1, stream));
        PSG_TRY(psg_net_geometry(n, starts, 1, stream));
    }
    PSG_TRY(psg_net_forward(n, t, nullptr, nullptr, stream));
    // f(outputs, labels) of nontarget.py:120-128 / target.py:149-168 and its gradient; `hit` feeds
    // the accuracy test of :86-87 / :96-105
    PSG_TRY(set_loss(n, 2, nullptr, b->labels, target, targeted_sign, kappa, s.f_rows, s.hit, st));
    PSG_TRY(psg_net_backward(n, t, nullptr, stream));
    if (neighbour > 0) {
        PSG_RUN(PF_LOSS, psg_nu_smooth_k(b->adv, b->images, C, N, neighbour, s.smooth_rows, s.smooth_grad, st));
    } else if (cudaMemsetAsync(s.smooth_rows, 0, 4 * (size_t)N * sizeof(float), st) != cudaSuccess) {
        return PSG_ECUDA;      // this rank does not own global block 0 (nontarget.py:131): no smoothness term
    }
    PSG_RUN(PF_LOSS, psg_nu_reduce_k(s.f_rows, s.l2_rows, s.smooth_rows, s.hit, b->mask, rows, N, c, step, acc_denom, thr,
                                     exit_above, count_masked_only, b->cost, b->status, st));
    PSG_RUN(PF_PGD, psg_nu_adam_k(b->w, b->adam_m, b->adam_v, g0, b->adv, b->images, s.smooth_grad, b->mask, B, C, N, fld, c,
                                  step_size, bc2_sqrt, 0.9f, 0.999f, 1e-8f, reset_adam, b->status, st));
    return PSG_OK;
}

extern "C" int psg_clamp(float *x, int64_t count, float lo, float hi, psg_stream_t stream)
{
    if (!x || count <= 0) return PSG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    PSG_RUN(PF_PGD, psg_clamp_k(x, count, lo, hi, st));
    return PSG_OK;
}

extern "C" int64_t psg_launch_count(void) { return g_psg_launch_count; }
extern "C" int psg_version(void) { return 100; }
