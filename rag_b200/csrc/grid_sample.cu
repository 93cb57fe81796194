// 4-D bilinear F.grid_sample, forward and fixed-order backward: the warp of a self-supervised stereo loss, which synthesises
// one view from the other and a predicted disparity (src_self/models/loss.py of the reference, inferred: SURVEY.md row 13).
//
// Contract: ATen's grid_sampler_2d for input [N,C,Hi,Wi] and grid [N,Ho,Wo,2], contiguous fp32, mode 'bilinear', padding
// 'zeros' or 'border', either align_corners.  The index arithmetic restates ATen's (aten/src/ATen/native/cuda/GridSampler.cuh),
// all fp32, per output sample (n, ho, wo) with grid value (gx, gy):
//     unnormalise:  align_corners:  i = ((g + 1) / 2) * (size - 1)      (d i / d g = (size - 1) / 2)
//                   otherwise:      i = ((g + 1) * size - 1) / 2        (d i / d g = size / 2)
//     border:       forward clips with min(size - 1, max(i, 0)); the backward clips with comparisons, and the clip's
//                   gradient is 0 where it clipped (i <= 0 or i >= size - 1).  The two differ only for NaN, as in ATen:
//                   max(NaN, 0) = 0 in the forward, NaN in the backward.
//     then i = -100 if i is not finite or outside [INT_MIN, INT_MAX - 1]   (every corner out of bounds)
//     corners  x0 = floor(ix), y0 = floor(iy): nw (x0,y0), ne (x0+1,y0), sw (x0,y0+1), se (x0+1,y0+1)
//     weights  nw = (x1 - ix)(y1 - iy), ne = (ix - x0)(y1 - iy), sw = (x1 - ix)(iy - y0), se = (ix - x0)(iy - y0)
//     out[n,c,ho,wo] = sum over the in-bounds corners, in the order nw, ne, sw, se, of in[n,c,y,x] * w
// The integer corner is clamped to [-2, size] before the bounds test: a grid value of any size (or NaN) reads nothing out of
// bounds, and every clamped corner stays out of bounds, so the result is ATen's.
//
// Forward: one thread per output sample, channels in a loop (loads of the grid and stores of the output coalesced along wo).
// Grid gradient: per sample over the channels in ascending order, as ATen; no atomics.
// Input gradient: ATen scatters with atomicAdd, so its sum order is the arrival order.  Here the order is defined:
//     gin[n,c,y,x] = sum of w * gout[n,c,ho,wo] over every (sample, corner) that references (y, x), in ascending flat sample
//     index (n*Ho + ho)*Wo + wo and within a sample in the corner order nw, ne, sw, se (fp32, fused multiply-add).
// It is built as (1) one entry per (sample, corner): key = flat input pixel (n*Hi + y)*Wi + x, or N*Hi*Wi when the corner is
// out of bounds, value = 4*sample + corner, and the corner's weight at index value; (2) a stable radix sort of the pairs by key
// (CUB DeviceRadixSort, sorting only the bits a key can have); since the values start in ascending order, each pixel's entries
// end up in the order above; (3) each pixel's segment [begin, end) marked from the sorted keys; (4) one thread per input pixel
// gathering its segment for every channel.  No float atomics anywhere; pixels that no sample references get a plain zero store.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace rag {

namespace {

constexpr int kGsThreads = 256;
constexpr int kGsChannels = 4;      // channels per pass of the gather kernel (registers per thread)
constexpr int kGsPtxVersion = 1000; // the PTX version the library is built for (compute_100a): selects CUB's tuning policy

using GsSort = cub::DispatchRadixSort<false, uint32_t, uint32_t, uint32_t>;

__device__ __forceinline__ float gs_unnormalize(float coord, int size, bool ac) {
    if (ac) return ((coord + 1.f) / 2) * (size - 1);
    return ((coord + 1.f) * size - 1) / 2;
}

__device__ __forceinline__ float gs_safe(float x) {
    if (x > (float)(INT_MAX - 1) || x < (float)INT_MIN || !isfinite(x)) return -100.f;
    return x;
}

// the forward's source index
__device__ __forceinline__ float gs_source(float coord, int size, bool border, bool ac) {
    float i = gs_unnormalize(coord, size, ac);
    if (border) i = fminf((float)(size - 1), fmaxf(i, 0.f));
    return gs_safe(i);
}

// the backward's source index and d index / d coord
__device__ __forceinline__ float gs_source_grad(float coord, int size, bool border, bool ac, float& mult) {
    mult = ac ? (float)(size - 1) / 2 : (float)size / 2;
    float i = gs_unnormalize(coord, size, ac);
    if (border) {
        if (i <= 0.f) {
            i = 0.f;
            mult = 0.f;
        } else if (i >= (float)(size - 1)) {
            i = (float)(size - 1);
            mult = 0.f;
        }
    }
    return gs_safe(i);
}

// floor, clamped to [-2, size]: outside that range every corner is out of bounds either way
__device__ __forceinline__ int gs_corner(float i, int size) { return (int)fminf(fmaxf(floorf(i), -2.f), (float)size); }

__device__ __forceinline__ bool gs_in(int y, int x, int H, int W) { return y >= 0 && y < H && x >= 0 && x < W; }

template <bool BORDER, bool AC>
__global__ void __launch_bounds__(kGsThreads)
grid_sample_fwd_kernel(const float* __restrict__ in, const float* __restrict__ grid, float* __restrict__ out, int N, int C, int Hi,
                       int Wi, int Ho, int Wo) {
    const int HWo = Ho * Wo, HWi = Hi * Wi;
    const int s = blockIdx.x * kGsThreads + threadIdx.x;
    if (s >= N * HWo) return;
    const int n = s / HWo, hw = s - n * HWo;
    const float2 g = __ldg(reinterpret_cast<const float2*>(grid) + s);
    const float ix = gs_source(g.x, Wi, BORDER, AC), iy = gs_source(g.y, Hi, BORDER, AC);
    const int x0 = gs_corner(ix, Wi), y0 = gs_corner(iy, Hi), x1 = x0 + 1, y1 = y0 + 1;
    const float nw = ((float)x1 - ix) * ((float)y1 - iy);
    const float ne = (ix - (float)x0) * ((float)y1 - iy);
    const float sw = ((float)x1 - ix) * (iy - (float)y0);
    const float se = (ix - (float)x0) * (iy - (float)y0);
    const bool bnw = gs_in(y0, x0, Hi, Wi), bne = gs_in(y0, x1, Hi, Wi), bsw = gs_in(y1, x0, Hi, Wi), bse = gs_in(y1, x1, Hi, Wi);
    const float* p = in + (size_t)n * C * HWi;
    float* o = out + (size_t)n * C * HWo + hw;
    for (int c = 0; c < C; ++c, p += HWi, o += HWo) {
        float acc = 0.f;
        if (bnw) acc += __ldg(p + y0 * Wi + x0) * nw;
        if (bne) acc += __ldg(p + y0 * Wi + x1) * ne;
        if (bsw) acc += __ldg(p + y1 * Wi + x0) * sw;
        if (bse) acc += __ldg(p + y1 * Wi + x1) * se;
        *o = acc;
    }
}

// One thread per output sample: the grid gradient (ggrid != NULL) and the sort entries of the input gradient (keys != NULL).
template <bool BORDER, bool AC>
__global__ void __launch_bounds__(kGsThreads)
grid_sample_bwd_sample_kernel(const float* __restrict__ gout, const float* __restrict__ in, const float* __restrict__ grid,
                              float* __restrict__ ggrid, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                              float* __restrict__ wts, int N, int C, int Hi, int Wi, int Ho, int Wo) {
    const int HWo = Ho * Wo, HWi = Hi * Wi;
    const int s = blockIdx.x * kGsThreads + threadIdx.x;
    if (s >= N * HWo) return;
    const int n = s / HWo, hw = s - n * HWo;
    const float2 g = __ldg(reinterpret_cast<const float2*>(grid) + s);
    float gx_mult, gy_mult;
    const float ix = gs_source_grad(g.x, Wi, BORDER, AC, gx_mult), iy = gs_source_grad(g.y, Hi, BORDER, AC, gy_mult);
    const int x0 = gs_corner(ix, Wi), y0 = gs_corner(iy, Hi), x1 = x0 + 1, y1 = y0 + 1;
    const float nw = ((float)x1 - ix) * ((float)y1 - iy);
    const float ne = (ix - (float)x0) * ((float)y1 - iy);
    const float sw = ((float)x1 - ix) * (iy - (float)y0);
    const float se = (ix - (float)x0) * (iy - (float)y0);
    const bool bnw = gs_in(y0, x0, Hi, Wi), bne = gs_in(y0, x1, Hi, Wi), bsw = gs_in(y1, x0, Hi, Wi), bse = gs_in(y1, x1, Hi, Wi);
    if (keys) {
        const uint32_t none = (uint32_t)N * (uint32_t)HWi, base = (uint32_t)n * (uint32_t)HWi;
        const uint4 k = make_uint4(bnw ? base + y0 * Wi + x0 : none, bne ? base + y0 * Wi + x1 : none,
                                   bsw ? base + y1 * Wi + x0 : none, bse ? base + y1 * Wi + x1 : none);
        const uint32_t v = 4u * (uint32_t)s;
        reinterpret_cast<uint4*>(keys)[s] = k;
        reinterpret_cast<uint4*>(vals)[s] = make_uint4(v, v + 1, v + 2, v + 3);
        reinterpret_cast<float4*>(wts)[s] = make_float4(nw, ne, sw, se);
    }
    if (ggrid) {
        float gix = 0.f, giy = 0.f;
        const float* p = in + (size_t)n * C * HWi;
        const float* go = gout + (size_t)n * C * HWo + hw;
        for (int c = 0; c < C; ++c, p += HWi, go += HWo) {
            const float gO = __ldg(go);
            if (bnw) {
                const float v = __ldg(p + y0 * Wi + x0);
                gix -= v * ((float)y1 - iy) * gO;
                giy -= v * ((float)x1 - ix) * gO;
            }
            if (bne) {
                const float v = __ldg(p + y0 * Wi + x1);
                gix += v * ((float)y1 - iy) * gO;
                giy -= v * (ix - (float)x0) * gO;
            }
            if (bsw) {
                const float v = __ldg(p + y1 * Wi + x0);
                gix -= v * (iy - (float)y0) * gO;
                giy += v * ((float)x1 - ix) * gO;
            }
            if (bse) {
                const float v = __ldg(p + y1 * Wi + x1);
                gix += v * (iy - (float)y0) * gO;
                giy += v * (ix - (float)x0) * gO;
            }
        }
        reinterpret_cast<float2*>(ggrid)[s] = make_float2(gx_mult * gix, gy_mult * giy);
    }
}

// seg_begin / seg_end [N*Hi*Wi] (zeroed before): the range of sorted entries of each referenced pixel
__global__ void __launch_bounds__(kGsThreads)
grid_sample_segments_kernel(const uint32_t* __restrict__ keys, int M, uint32_t none, int* __restrict__ seg_begin,
                            int* __restrict__ seg_end) {
    const int i = blockIdx.x * kGsThreads + threadIdx.x;
    if (i >= M) return;
    const uint32_t k = keys[i];
    if (k >= none) return;
    if (i == 0 || keys[i - 1] != k) seg_begin[k] = i;
    if (i == M - 1 || keys[i + 1] != k) seg_end[k] = i + 1;
}

// One thread per input pixel: gin[n,c,y,x] = sum over its segment, in order, of w * gout[n,c,sample], kGsChannels at a time.
__global__ void __launch_bounds__(kGsThreads)
grid_sample_gather_kernel(const float* __restrict__ gout, const uint32_t* __restrict__ vals, const float* __restrict__ wts,
                          const int* __restrict__ seg_begin, const int* __restrict__ seg_end, float* __restrict__ gin, int N,
                          int C, int HWi, int HWo) {
    const int p = blockIdx.x * kGsThreads + threadIdx.x;
    if (p >= N * HWi) return;
    const int n = p / HWi, yx = p - n * HWi;
    const int b = seg_begin[p], e = seg_end[p];
    // gout[n, c, hw] = gout[sample + (n*(C-1) + c) * HWo] for sample = n*HWo + hw
    const float* go = gout + (size_t)n * (C - 1) * HWo;
    float* gi = gin + (size_t)n * C * HWi + yx;
    for (int c0 = 0; c0 < C; c0 += kGsChannels) {
        float acc[kGsChannels] = {};
        const int nc = min(kGsChannels, C - c0);
        for (int i = b; i < e; ++i) {
            const uint32_t v = __ldg(vals + i);
            const float w = __ldg(wts + v);
            const float* q = go + (size_t)c0 * HWo + (v >> 2);
#pragma unroll
            for (int j = 0; j < kGsChannels; ++j)
                if (j < nc) acc[j] = fmaf(w, __ldg(q + (size_t)j * HWo), acc[j]);
        }
#pragma unroll
        for (int j = 0; j < kGsChannels; ++j)
            if (j < nc) gi[(size_t)(c0 + j) * HWi] = acc[j];
    }
}

// host side ------------------------------------------------------------------------------------------------------------------

constexpr size_t kGsAlign = 256;

size_t gs_up(size_t b) { return (b + kGsAlign - 1) / kGsAlign * kGsAlign; }

int gs_key_bits(long long none) {
    int bits = 1;
    while (bits < 32 && (1ll << bits) <= none) ++bits;
    return bits;
}

// Shape limits: every flat index and entry count below 2^31.  Host-only; no CUDA call.
int gs_check_shape(const char* who, int N, int C, int Hi, int Wi, int Ho, int Wo) {
    if (N <= 0 || C <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    const long long lim = 1ll << 31;
    const long long S = (long long)N * Ho * Wo, P = (long long)N * Hi * Wi;
    if (4 * S >= lim || P >= lim || (long long)C * P >= lim || (long long)C * S >= lim)
        return fail(RAG_E_SHAPE, "%s: a flat index or the entry count 4*N*Ho*Wo reaches 2^31", who);
    return RAG_OK;
}

struct GsLayout {
    size_t keys[2], vals[2], wts, seg, sort, sort_bytes, total;
};

// Workspace of the input gradient: keys, values (both double-buffered) and weights per sample-corner, begin and end per input
// pixel, then CUB's sort storage.  Each region starts 256-byte aligned.  sort_bytes is computed without a device, for the
// tuning policy of compute_100a (the only code in the library), so a query works on any host.
int gs_layout(int N, int Hi, int Wi, int Ho, int Wo, GsLayout& L) {
    const size_t M = (size_t)4 * N * Ho * Wo, P = (size_t)N * Hi * Wi;
    size_t at = 0;
    for (int i = 0; i < 2; ++i) { L.keys[i] = at; at += gs_up(M * 4); }
    for (int i = 0; i < 2; ++i) { L.vals[i] = at; at += gs_up(M * 4); }
    L.wts = at; at += gs_up(M * 4);
    L.seg = at; at += gs_up(P * 8);
    L.sort = at;
    cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
    size_t bytes = 0;
    GsSort d(nullptr, bytes, k, v, (uint32_t)M, 0, gs_key_bits((long long)P), true, nullptr, kGsPtxVersion);
    const cudaError_t e = GsSort::max_policy_t::Invoke(kGsPtxVersion, d);
    if (e != cudaSuccess) return fail((int)e, "grid_sample_bwd_workspace_bytes: sort size query: %s", cudaGetErrorString(e));
    L.sort_bytes = bytes;
    L.total = at + gs_up(bytes);
    return RAG_OK;
}

}  // namespace

int grid_sample_fwd(const float* in, const float* grid, float* out, int N, int C, int Hi, int Wi, int Ho, int Wo, int padding_mode,
                    int align_corners, cudaStream_t st) {
    const char* who = "grid_sample_fwd";
    if (!in || !grid || !out) return fail(RAG_E_NULL, "%s: null pointer", who);
    if (int e = gs_check_shape(who, N, C, Hi, Wi, Ho, Wo)) return e;
    if (padding_mode != 0 && padding_mode != 1) return fail(RAG_E_SHAPE, "%s: padding_mode must be 0 (zeros) or 1 (border)", who);
    if (!aligned(in, 4) || !aligned(out, 4) || !aligned(grid, 8)) return fail(RAG_E_ALIGN, "%s: in / out 4-byte, grid 8-byte aligned", who);
    const unsigned blocks = (unsigned)(((long long)N * Ho * Wo + kGsThreads - 1) / kGsThreads);
    auto kern = padding_mode ? (align_corners ? grid_sample_fwd_kernel<true, true> : grid_sample_fwd_kernel<true, false>)
                             : (align_corners ? grid_sample_fwd_kernel<false, true> : grid_sample_fwd_kernel<false, false>);
    kern<<<blocks, kGsThreads, 0, st>>>(in, grid, out, N, C, Hi, Wi, Ho, Wo);
    return check_launch(who);
}

size_t grid_sample_bwd_workspace_bytes(int N, int C, int Hi, int Wi, int Ho, int Wo) {
    if (gs_check_shape("grid_sample_bwd_workspace_bytes", N, C, Hi, Wi, Ho, Wo)) return 0;
    GsLayout L;
    if (gs_layout(N, Hi, Wi, Ho, Wo, L)) return 0;
    return L.total;
}

int grid_sample_bwd(const float* gout, const float* in, const float* grid, float* gin, float* ggrid, void* workspace,
                    size_t workspace_bytes, int N, int C, int Hi, int Wi, int Ho, int Wo, int padding_mode, int align_corners,
                    cudaStream_t st) {
    const char* who = "grid_sample_bwd";
    if (!gout || !grid || (ggrid && !in) || (gin && !workspace)) return fail(RAG_E_NULL, "%s: null pointer", who);
    if (int e = gs_check_shape(who, N, C, Hi, Wi, Ho, Wo)) return e;
    if (padding_mode != 0 && padding_mode != 1) return fail(RAG_E_SHAPE, "%s: padding_mode must be 0 (zeros) or 1 (border)", who);
    if (!aligned(gout, 4) || (in && !aligned(in, 4)) || (gin && !aligned(gin, 4)) || !aligned(grid, 8) || (ggrid && !aligned(ggrid, 8)) ||
        (workspace && !aligned(workspace, kGsAlign)))
        return fail(RAG_E_ALIGN, "%s: gout / in / gin 4-byte, grid / ggrid 8-byte, workspace 256-byte aligned", who);
    GsLayout L{};
    if (gin) {
        if (int e = gs_layout(N, Hi, Wi, Ho, Wo, L)) return e;
        if (workspace_bytes < L.total)
            return fail(RAG_E_SHAPE, "%s: workspace of %zu bytes, need %zu (rag_grid_sample_bwd_workspace_bytes)", who, workspace_bytes, L.total);
    }
    if (!gin && !ggrid) return RAG_OK;
    const int S = N * Ho * Wo, M = 4 * S, P = N * Hi * Wi;
    char* ws = static_cast<char*>(workspace);
    uint32_t* keys0 = gin ? reinterpret_cast<uint32_t*>(ws + L.keys[0]) : nullptr;
    uint32_t* vals0 = gin ? reinterpret_cast<uint32_t*>(ws + L.vals[0]) : nullptr;
    float* wts = gin ? reinterpret_cast<float*>(ws + L.wts) : nullptr;
    const unsigned blocks = (unsigned)((S + kGsThreads - 1) / kGsThreads);
    auto kern = padding_mode ? (align_corners ? grid_sample_bwd_sample_kernel<true, true> : grid_sample_bwd_sample_kernel<true, false>)
                             : (align_corners ? grid_sample_bwd_sample_kernel<false, true> : grid_sample_bwd_sample_kernel<false, false>);
    kern<<<blocks, kGsThreads, 0, st>>>(gout, in, grid, ggrid, keys0, vals0, wts, N, C, Hi, Wi, Ho, Wo);
    if (int e = check_launch("grid_sample_bwd(samples)")) return e;
    if (!gin) return RAG_OK;

    cub::DoubleBuffer<uint32_t> keys(keys0, reinterpret_cast<uint32_t*>(ws + L.keys[1]));
    cub::DoubleBuffer<uint32_t> vals(vals0, reinterpret_cast<uint32_t*>(ws + L.vals[1]));
    size_t sort_bytes = 0;
    cudaError_t e = GsSort::Dispatch(nullptr, sort_bytes, keys, vals, (uint32_t)M, 0, gs_key_bits(P), true, st);
    if (e == cudaSuccess && sort_bytes > L.sort_bytes)
        return fail(RAG_E_SHAPE, "%s: the device's sort needs %zu bytes, the workspace holds %zu", who, sort_bytes, L.sort_bytes);
    if (e == cudaSuccess) e = GsSort::Dispatch(ws + L.sort, sort_bytes, keys, vals, (uint32_t)M, 0, gs_key_bits(P), true, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ws + L.seg, 0, (size_t)P * 8, st);
    if (e != cudaSuccess) return fail((int)e, "%s: sort: %s", who, cudaGetErrorString(e));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    int* seg_begin = reinterpret_cast<int*>(ws + L.seg);
    grid_sample_segments_kernel<<<(unsigned)((M + kGsThreads - 1) / kGsThreads), kGsThreads, 0, st>>>(keys.Current(), M, (uint32_t)P,
                                                                                                      seg_begin, seg_begin + P);
    if (int e2 = check_launch("grid_sample_bwd(segments)")) return e2;
    grid_sample_gather_kernel<<<(unsigned)((P + kGsThreads - 1) / kGsThreads), kGsThreads, 0, st>>>(
        gout, vals.Current(), wts, seg_begin, seg_begin + P, gin, N, C, Hi * Wi, Ho * Wo);
    return check_launch("grid_sample_bwd(gather)");
}

}  // namespace rag
