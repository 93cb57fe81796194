// The Matching Net's pointwise layers: ConvBR_3d(C, O, 1, 1, 0) = bias-free 1x1x1 Conv3d C -> O, then BatchNorm3d + ReLU
// (src/automl/operations_3d.py:31-47) -- `last_12_3d` (48 -> 24), `last_6_3d` (24 -> 12) and, inferred, the cells' 1x1x1
// preprocessing layers.  With x [B,C,S] (S = D*H*W) and w [O,C]:
//     z[b,o,s]   = sum_c w[o,c] x[b,c,s]                                      (forward, c ascending)
//     gin[b,c,s] = sum_o w[o,c] gz[b,o,s]                                     (data gradient, o ascending)
//     gw[o,c]    = sum_{b,s} gz[b,o,s] x[b,c,s]                               (weight gradient)
// (C, O) are run-time values, 1 <= C <= 64 and 1 <= O <= 32; the kernels are instantiated for the output tile OT = O rounded
// up to a multiple of 4 (the weights of the missing outputs are zero in shared memory and their stores are skipped).
//
// These layers do ~C*O MAC per (C + O) * 4 bytes of a voxel: HBM traffic bounds them.  Forward: a thread owns 4 consecutive
// voxels for all OT outputs (4*OT accumulators), reads x once with 128-bit loads and writes out once with streamed 128-bit
// stores; the weights sit in shared memory as [c][o] (one LDS.128 broadcast per four outputs and input channel).
//
// Fused backward, from the upstream gradient g, the saved z and bn3d's [O,7] consts: the gradient at the convolution output,
// gz = a (g' - m1 - zh m2) (bn3d.cuh, the expression bn3d_bwd_gz_kernel uses), is formed in registers and never written.  A
// fixed grid (148 x the CTAs per SM its shared memory allows, a function of (C, O)) walks tiles of kPwNV voxels (tile
// blockIdx.x, blockIdx.x + G, ...).  Per tile, a thread owns 2 voxels: it forms their gz for all outputs and writes gin
// from them (weights as [c][o] in shared memory).  For the weight gradient the CTA parks gz and x of the tile in shared
// memory, four channels per float4; a thread owns a 4 (o) x 4 (c) block of gw and every R-th voxel of the tile (R = 128 /
// number of blocks replicas of the block grid, so small layers keep all threads busy).  A CTA keeps its sums across all its
// tiles.  The replicas are added in a fixed order into one fp32 partial per CTA and (o, c); a final kernel adds the
// partials in fp64 in a fixed order: bitwise repeatable.  No constant memory, no atomics: stateless and capturable.
#include <algorithm>
#include <climits>

#include "bn3d.cuh"
#include "common.cuh"

namespace rag {

constexpr int kPwThreads = 128;
constexpr int kPwMaxC = 64, kPwMaxO = 32;
constexpr int kPwNV = 256;                // voxels per backward tile (2 per thread)
constexpr int kPwRow = kPwNV + 1;         // float4 row stride of the tile: neighbouring rows land 16 bytes apart in the banks
constexpr int kPwGridSMs = 148;           // the backward's grid: kPwGridSMs * pw_ctas_per_sm(C, O) CTAs (= partials per weight),
                                          // a function of (C, O) only, so the sums are repeatable on any device

// grid: x = ceil(S/4 / 128), y = B; 128 threads.  smem: C * OT floats.  OT = 28 / 32 are held to 3 CTAs (12 warps) per SM,
// 168 registers: left alone they take 221 / 186 and fit 2, and a streaming kernel wants the loads of more warps in flight.
// No spills.  Smaller tiles fit 3 or more CTAs as compiled without the hint (0 = none).
template <int OT>
__global__ void __launch_bounds__(kPwThreads, OT >= 28 ? 3 : 0)
conv3d_pw_fwd_kernel(const float4* __restrict__ in, const float* __restrict__ w, const float* __restrict__ scale,
                     const float* __restrict__ shift, int relu, float4* __restrict__ out, int C, int O, size_t S4) {
    extern __shared__ __align__(16) float pw_smem[];
    for (int i = threadIdx.x; i < C * OT; i += kPwThreads) {      // [c][o], zero for o >= O
        const int c = i / OT, o = i - c * OT;
        pw_smem[i] = o < O ? __ldg(w + (size_t)o * C + c) : 0.f;
    }
    __syncthreads();
    const size_t q = (size_t)blockIdx.x * kPwThreads + threadIdx.x;
    if (q >= S4) return;
    const int b = blockIdx.y;
    const float4* xp = in + (size_t)b * C * S4 + q;
    const float4* ws = reinterpret_cast<const float4*>(pw_smem);
    float acc[OT][4];
#pragma unroll
    for (int o = 0; o < OT; ++o)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[o][j] = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
        const float4 xv = ld_stream(xp + (size_t)c * S4);
#pragma unroll
        for (int g = 0; g < OT / 4; ++g) {
            const float4 wv = ws[c * (OT / 4) + g];
            acc[4 * g + 0][0] = __fmaf_rn(wv.x, xv.x, acc[4 * g + 0][0]); acc[4 * g + 0][1] = __fmaf_rn(wv.x, xv.y, acc[4 * g + 0][1]);
            acc[4 * g + 0][2] = __fmaf_rn(wv.x, xv.z, acc[4 * g + 0][2]); acc[4 * g + 0][3] = __fmaf_rn(wv.x, xv.w, acc[4 * g + 0][3]);
            acc[4 * g + 1][0] = __fmaf_rn(wv.y, xv.x, acc[4 * g + 1][0]); acc[4 * g + 1][1] = __fmaf_rn(wv.y, xv.y, acc[4 * g + 1][1]);
            acc[4 * g + 1][2] = __fmaf_rn(wv.y, xv.z, acc[4 * g + 1][2]); acc[4 * g + 1][3] = __fmaf_rn(wv.y, xv.w, acc[4 * g + 1][3]);
            acc[4 * g + 2][0] = __fmaf_rn(wv.z, xv.x, acc[4 * g + 2][0]); acc[4 * g + 2][1] = __fmaf_rn(wv.z, xv.y, acc[4 * g + 2][1]);
            acc[4 * g + 2][2] = __fmaf_rn(wv.z, xv.z, acc[4 * g + 2][2]); acc[4 * g + 2][3] = __fmaf_rn(wv.z, xv.w, acc[4 * g + 2][3]);
            acc[4 * g + 3][0] = __fmaf_rn(wv.w, xv.x, acc[4 * g + 3][0]); acc[4 * g + 3][1] = __fmaf_rn(wv.w, xv.y, acc[4 * g + 3][1]);
            acc[4 * g + 3][2] = __fmaf_rn(wv.w, xv.z, acc[4 * g + 3][2]); acc[4 * g + 3][3] = __fmaf_rn(wv.w, xv.w, acc[4 * g + 3][3]);
        }
    }
    float4* op = out + (size_t)b * O * S4 + q;
#pragma unroll
    for (int o = 0; o < OT; ++o) {
        if (o < O) {
            float4 r = make_float4(acc[o][0], acc[o][1], acc[o][2], acc[o][3]);
            if (scale) {
                const float sc = __ldg(scale + o), sh = __ldg(shift + o);
                r.x = __fmaf_rn(r.x, sc, sh); r.y = __fmaf_rn(r.y, sc, sh); r.z = __fmaf_rn(r.z, sc, sh); r.w = __fmaf_rn(r.w, sc, sh);
            }
            if (relu) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
            st_stream(op + (size_t)o * S4, r);
        }
    }
}

__host__ __device__ constexpr int pw_cb(int C) { return (C + 3) / 4; }      // float4 channel groups of x

// smem floats of the backward: consts [OT][7] | w [C][OT] | x tile [CB][kPwRow] float4 | gz tile [OT/4][kPwRow] float4
__host__ __device__ constexpr size_t pw_bwd_smem_floats(int C, int OT) {
    return (size_t)((OT * 7 + C * OT + 3) / 4 * 4) + 4 * (size_t)(pw_cb(C) + OT / 4) * kPwRow;
}

// resident CTAs per SM the backward is sized for: what 200 KB of shared memory holds, 1..6
__host__ __device__ constexpr int pw_ctas_per_sm(int C, int O) {
    const int n = (int)(200 * 1024 / (4 * pw_bwd_smem_floats(C, (O + 3) / 4 * 4)));
    return n < 1 ? 1 : n > 6 ? 6 : n;
}
__host__ __device__ constexpr int pw_groups(int C, int O) { return kPwGridSMs * pw_ctas_per_sm(C, O); }

// grid G (<= pw_groups(C, O)), 128 threads.  gin (nullable) [B,C,S]; part (nullable) [G][O][C].  S2 = S/2; n_st = ceil(S/kPwNV).
template <int OT>
__global__ void __launch_bounds__(kPwThreads)
conv3d_pw_bwd_kernel(const float2* __restrict__ g, const float2* __restrict__ z, const float* __restrict__ consts,
                     const float2* __restrict__ in, const float* __restrict__ w, float2* __restrict__ gin, float* __restrict__ part,
                     int C, int O, size_t S2, int n_st, long long n_tiles) {
    extern __shared__ __align__(16) float pw_smem[];
    float* cs = pw_smem;                                          // [OT][7], a = 0 for o >= O: gz = 0 there
    float* wsm = cs + OT * 7;                                     // [c][o]
    float4* xs = reinterpret_cast<float4*>(pw_smem + (OT * 7 + C * OT + 3) / 4 * 4);
    float4* gs = xs + (size_t)pw_cb(C) * kPwRow;
    const int tid = threadIdx.x, CB = pw_cb(C);
    for (int i = tid; i < OT * 7; i += kPwThreads) cs[i] = i < O * 7 ? __ldg(consts + i) : 0.f;
    if (gin)
        for (int i = tid; i < C * OT; i += kPwThreads) {
            const int c = i / OT, o = i - c * OT;
            wsm[i] = o < O ? __ldg(w + (size_t)o * C + c) : 0.f;
        }
    __syncthreads();

    // the thread's 4 (o) x 4 (c) block of the weight gradient and its replica: R = 128 / NBLK copies of the block grid each
    // take every R-th voxel of a tile, and are added in replica order at the end
    const int NBLK = CB * (OT / 4), R = kPwThreads / NBLK;
    const int rep = tid / NBLK;
    const bool owner = rep < R;
    const int blk = tid - rep * NBLK, cb = owner ? blk % CB : 0, ob = owner ? blk / CB : 0;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[i][k] = 0.f;

#pragma unroll 1
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int b = (int)(t / n_st), st = (int)(t - (long long)b * n_st);
        const size_t v2 = (size_t)st * (kPwNV / 2) + tid;         // the thread's voxel pair
        const bool valid = v2 < S2;
        float gz[OT][2];
#pragma unroll
        for (int o = 0; o < OT; ++o) {
            gz[o][0] = gz[o][1] = 0.f;
            if (o < O && valid) {
                const size_t idx = ((size_t)b * O + o) * S2 + v2;
                const float2 gv = ld_stream(g + idx), zv = ld_stream(z + idx);
                const float* k = cs + 7 * o;
                gz[o][0] = bn3d_gz(gv.x, zv.x, k[0], k[1], k[2], k[3], k[4], k[5], k[6]);
                gz[o][1] = bn3d_gz(gv.y, zv.y, k[0], k[1], k[2], k[3], k[4], k[5], k[6]);
            }
        }
        if (gin && valid) {
            const float4* w4 = reinterpret_cast<const float4*>(wsm);
#pragma unroll 2
            for (int c = 0; c < C; ++c) {
                float2 r = make_float2(0.f, 0.f);
#pragma unroll
                for (int q = 0; q < OT / 4; ++q) {
                    const float4 wv = w4[c * (OT / 4) + q];
                    r.x = __fmaf_rn(wv.x, gz[4 * q][0], r.x); r.y = __fmaf_rn(wv.x, gz[4 * q][1], r.y);
                    r.x = __fmaf_rn(wv.y, gz[4 * q + 1][0], r.x); r.y = __fmaf_rn(wv.y, gz[4 * q + 1][1], r.y);
                    r.x = __fmaf_rn(wv.z, gz[4 * q + 2][0], r.x); r.y = __fmaf_rn(wv.z, gz[4 * q + 2][1], r.y);
                    r.x = __fmaf_rn(wv.w, gz[4 * q + 3][0], r.x); r.y = __fmaf_rn(wv.w, gz[4 * q + 3][1], r.y);
                }
                st_stream(gin + ((size_t)b * C + c) * S2 + v2, r);
            }
        }
        if (part) {
            __syncthreads();                                      // the previous tile's blocks are done with the tile buffers
#pragma unroll
            for (int q = 0; q < OT / 4; ++q) {
                gs[q * kPwRow + 2 * tid] = make_float4(gz[4 * q][0], gz[4 * q + 1][0], gz[4 * q + 2][0], gz[4 * q + 3][0]);
                gs[q * kPwRow + 2 * tid + 1] = make_float4(gz[4 * q][1], gz[4 * q + 1][1], gz[4 * q + 2][1], gz[4 * q + 3][1]);
            }
            for (int q = 0; q < CB; ++q) {
                float2 xv[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = 4 * q + k;
                    xv[k] = (c < C && valid) ? ld_stream(in + ((size_t)b * C + c) * S2 + v2) : make_float2(0.f, 0.f);
                }
                xs[q * kPwRow + 2 * tid] = make_float4(xv[0].x, xv[1].x, xv[2].x, xv[3].x);
                xs[q * kPwRow + 2 * tid + 1] = make_float4(xv[0].y, xv[1].y, xv[2].y, xv[3].y);
            }
            __syncthreads();
            if (owner) {
                const float4* xr = xs + cb * kPwRow;
                const float4* gr = gs + ob * kPwRow;
#pragma unroll 4
                for (int v = rep; v < kPwNV; v += R) {
                    const float4 xv = xr[v], gv = gr[v];
                    const float gg[4] = {gv.x, gv.y, gv.z, gv.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int k = 0; k < 4; ++k) acc[i][k] = __fmaf_rn(gg[i], xx[k], acc[i][k]);
                }
            }
        }
    }
    if (!part) return;
    // replicas -> one partial per (o, c), r ascending; the tile buffers (>= 2 * 4 * kPwRow floats) hold the 128 x 16 sums
    float* red = reinterpret_cast<float*>(xs);
    __syncthreads();
    if (owner)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) red[(rep * NBLK + blk) * 16 + i * 4 + k] = acc[i][k];
    __syncthreads();
    float* pp = part + (size_t)blockIdx.x * O * C;
    for (int j = tid; j < NBLK * 16; j += kPwThreads) {
        const int bk = j >> 4, i = (j >> 2) & 3, k = j & 3;
        const int o = 4 * (bk / CB) + i, c = 4 * (bk % CB) + k;
        float a = 0.f;
        for (int r = 0; r < R; ++r) a += red[(r * NBLK + bk) * 16 + (j & 15)];
        if (o < O && c < C) pp[o * C + c] = a;
    }
}

// gw[i] = sum_g part[g][i], g ascending, fp64
__global__ void __launch_bounds__(256) conv3d_pw_wgrad_final_kernel(const float* __restrict__ part, float* __restrict__ gw, int n, int G) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double a = 0.0;
    for (int k = 0; k < G; ++k) a += (double)part[(size_t)k * n + i];
    gw[i] = (float)a;
}

// ---- host ---------------------------------------------------------------------------------------------------------------
static bool pw_in_range(int B, int C, int O, int D, int H, int W) {
    if (B <= 0 || C < 1 || C > kPwMaxC || O < 1 || O > kPwMaxO || D <= 0 || H <= 0 || W <= 0 || B > 65535) return false;
    const long long S = (long long)D * H * W;
    return S % 4 == 0 && (S + kPwNV - 1) / kPwNV <= INT_MAX;     // tiles per batch item (and the forward's grid.x) fit an int
}

static int pw_check(const char* who, int B, int C, int O, int D, int H, int W) {
    if (B <= 0 || C <= 0 || O <= 0 || D <= 0 || H <= 0 || W <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    if (!pw_in_range(B, C, O, D, H, W))
        return fail(RAG_E_SHAPE, "%s: needs 1 <= C <= %d, 1 <= O <= %d, B <= 65535 and D*H*W %% 4 == 0 (got B=%d C=%d O=%d D=%d H=%d W=%d)",
                    who, kPwMaxC, kPwMaxO, B, C, O, D, H, W);
    return RAG_OK;
}

template <int OT>
static int pw_launch_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                         int B, int C, int O, size_t S4, cudaStream_t st) {
    const size_t smem = (size_t)C * OT * sizeof(float);
    conv3d_pw_fwd_kernel<OT><<<dim3((unsigned)((S4 + kPwThreads - 1) / kPwThreads), B), kPwThreads, smem, st>>>(
        reinterpret_cast<const float4*>(in), w, scale, shift, relu, reinterpret_cast<float4*>(out), C, O, S4);
    return check_launch("conv3d_pw_fwd");
}

template <int OT>
static int pw_launch_bwd(const float* g, const float* z, const float* consts, const float* in, const float* w, float* gin, float* gw,
                         float* part, int B, int C, int O, long long S, cudaStream_t st) {
    const int n_st = (int)((S + kPwNV - 1) / kPwNV);
    const long long n_tiles = (long long)B * n_st;
    const int G = (int)std::min<long long>(pw_groups(C, O), n_tiles);   // a function of the shape only: repeatable on any device
    auto k = conv3d_pw_bwd_kernel<OT>;
    const size_t smem = pw_bwd_smem_floats(C, OT) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d_pw_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    k<<<G, kPwThreads, smem, st>>>(reinterpret_cast<const float2*>(g), reinterpret_cast<const float2*>(z), consts,
                                   reinterpret_cast<const float2*>(in), w, reinterpret_cast<float2*>(gin), gw ? part : nullptr,
                                   C, O, (size_t)(S / 2), n_st, n_tiles);
    if (int rc = check_launch("conv3d_pw_bwd")) return rc;
    if (!gw) return RAG_OK;
    const int n = O * C;
    conv3d_pw_wgrad_final_kernel<<<(n + 255) / 256, 256, 0, st>>>(part, gw, n, G);
    return check_launch("conv3d_pw_bwd(weight final)");
}

#define RAG_PW_DISPATCH(O, CALL)                         \
    switch ((O + 3) / 4) {                               \
        case 1: return CALL(4);                          \
        case 2: return CALL(8);                          \
        case 3: return CALL(12);                         \
        case 4: return CALL(16);                         \
        case 5: return CALL(20);                         \
        case 6: return CALL(24);                         \
        case 7: return CALL(28);                         \
        default: return CALL(32);                        \
    }

int conv3d_pw_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                  int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!in || !w || !out || (scale == nullptr) != (shift == nullptr)) return fail(RAG_E_NULL, "conv3d_pw_fwd: null pointer (scale and shift go together)");
    if (int rc = pw_check("conv3d_pw_fwd", B, C, O, D, H, W)) return rc;
    if (!aligned(in, 16) || !aligned(out, 16) || !aligned(w, 4) || (scale && (!aligned(scale, 4) || !aligned(shift, 4))))
        return fail(RAG_E_ALIGN, "conv3d_pw_fwd: in/out must be 16-byte aligned");
    const size_t S4 = (size_t)D * H * W / 4;
#define RAG_PW_FWD(OT) pw_launch_fwd<OT>(in, w, scale, shift, relu, out, B, C, O, S4, st)
    RAG_PW_DISPATCH(O, RAG_PW_FWD)
#undef RAG_PW_FWD
}

size_t conv3d_pw_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W) {
    if (!pw_in_range(B, C, O, D, H, W)) return 0;
    return (size_t)pw_groups(C, O) * O * C * sizeof(float);
}

int conv3d_pw_bwd(const float* g, const float* z, const float* consts, const float* in, const float* w, float* gin, float* gw,
                  float* workspace, int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!g || !z || !consts || (gin && !w) || (gw && (!in || !workspace))) return fail(RAG_E_NULL, "conv3d_pw_bwd: null pointer");
    if (int rc = pw_check("conv3d_pw_bwd", B, C, O, D, H, W)) return rc;
    if (!aligned(g, 16) || !aligned(z, 16) || !aligned(consts, 4) || (in && !aligned(in, 16)) || (gin && !aligned(gin, 16)) ||
        (w && !aligned(w, 4)) || (workspace && !aligned(workspace, 4)))
        return fail(RAG_E_ALIGN, "conv3d_pw_bwd: g/z/in/gin must be 16-byte aligned");
    if (!gin && !gw) return RAG_OK;
    const long long S = (long long)D * H * W;
#define RAG_PW_BWD(OT) pw_launch_bwd<OT>(g, z, consts, in, w, gin, gw, workspace, B, C, O, S, st)
    RAG_PW_DISPATCH(O, RAG_PW_BWD)
#undef RAG_PW_BWD
}

#undef RAG_PW_DISPATCH

}  // namespace rag
