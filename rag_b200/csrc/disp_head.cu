// Disparity head: trilinear x3 upsample -> softmin over D -> soft-argmin, fused, fwd + bwd (sm_100a).
//
// Reference semantics: src/models/rag_model.py:32-44 (Disp.forward) + :18-29 (DisparityRegression):
//   v = F.interpolate(cost_lr, [maxdisp, 3Hl, 3Wl], 'trilinear', align_corners=False)
//   disp = sum_k k * softmax_k(-v)
// The reference materialises the [B,maxdisp,H,W] volume about nine times (~1.1 GB/pair at 288x576);
// here the full-resolution volume never exists: the forward reads cost_lr once and writes disp (+2
// stats planes for the backward), the backward re-derives p_k from cost_lr and the stats.
//
// The upsample arithmetic replicates PyTorch's fp32 source-index / lambda computation
// (ATen/native/cuda/UpSample.cuh:115-130; nesting W -> H -> D as in UpSampleTrilinear3d.cu), because
// "ideal" 1/3, 2/3 weights are off by up to 1.3e-6 and move ~5% of pixels by more than 1e-4 px.
//
// Softmax numerics: exponents are taken in the log2 domain, z_k = -log2(e) * v_k, relative to a
// per-pixel reference exponent m that is only moved when the running maximum exceeds it by more
// than kTau (lazy rescaling, exact); sums are kept in short fp32 group accumulators that are
// folded into fp64 totals every 8 low-res bins, and the regression is centred (disp = kc +
// sum e_k (k-kc) / sum e_k), which keeps the kernel's own error ~1e-5 px -- an order of magnitude
// below the reference's fp32 noise floor (SURVEY.md section 8a H-1).
//
// Bound: NOT HBM. Per output pixel the head needs maxdisp exp2 on the SFU (16 lanes/clk/SM): 192
// MUFU.EX2 per pixel = 8 SMSP-clk per pixel-bin, which is the floor of this kernel (~7 us per
// 288x576 pair); the x3 kernel is organised so that everything else (blend, sums) fits under it.
#include <algorithm>

#include "common.cuh"

namespace rag {

constexpr float kNegLog2e = -1.4426950408889634f;


// ---------------------------------------------------------------------------------------------
// debug: the upsample alone
// ---------------------------------------------------------------------------------------------
template <bool FMA>
__global__ void upsample_kernel(const float* __restrict__ cost, float* __restrict__ out,
                                int Dl, int Hl, int Wl, int D, float sd, float sh, float sw) {
    const int H = 3 * Hl, W = 3 * Wl;
    const size_t n = (size_t)D * H * W;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const int b = blockIdx.y;
    const int w = idx % W, h = (idx / W) % H, k = idx / ((size_t)W * H);
    int t0, t1, h0, h1, w0, w1;
    float tl0, tl1, hl0, hl1, wl0, wl1;
    src_index<FMA>(sd, k, Dl, t0, t1, tl0, tl1);
    src_index<FMA>(sh, h, Hl, h0, h1, hl0, hl1);
    src_index<FMA>(sw, w, Wl, w0, w1, wl0, wl1);
    const float* s = cost + (size_t)b * Dl * Hl * Wl;
    auto at = [&](int t, int y, int x) { return s[((size_t)t * Hl + y) * Wl + x]; };
    const float v = tl0 * (hl0 * (wl0 * at(t0, h0, w0) + wl1 * at(t0, h0, w1)) + hl1 * (wl0 * at(t0, h1, w0) + wl1 * at(t0, h1, w1))) +
                    tl1 * (hl0 * (wl0 * at(t1, h0, w0) + wl1 * at(t1, h0, w1)) + hl1 * (wl0 * at(t1, h1, w0) + wl1 * at(t1, h1, w1)));
    out[(size_t)b * n + idx] = v;
}

// ---------------------------------------------------------------------------------------------
// generic forward: any (Dl, maxdisp); one thread per output pixel.  Slow path / cross-check.
// ---------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT)
head_fwd_generic_kernel(const float* __restrict__ cost, float* __restrict__ disp, float* __restrict__ stats,
                        int Dl, int Hl, int Wl, int D, float sd, float sh, float sw) {
    const int H = 3 * Hl, W = 3 * Wl;
    const int idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= H * W) return;
    const int b = blockIdx.y;
    const int h = idx / W, w = idx - h * W;
    int h0, h1, w0, w1;
    float hl0, hl1, wl0, wl1;
    src_index<true>(sh, h, Hl, h0, h1, hl0, hl1);
    src_index<true>(sw, w, Wl, w0, w1, wl0, wl1);
    const float* base = cost + (size_t)b * Dl * Hl * Wl;
    const int o00 = h0 * Wl + w0, o01 = h0 * Wl + w1, o10 = h1 * Wl + w0, o11 = h1 * Wl + w1;
    auto blend = [&](int j) {
        const float* s = base + (size_t)j * Hl * Wl;
        return hl0 * (wl0 * __ldg(s + o00) + wl1 * __ldg(s + o01)) + hl1 * (wl0 * __ldg(s + o10) + wl1 * __ldg(s + o11));
    };
    int cur = -1;
    float a0 = 0.f, a1 = 0.f;
    float m = -INFINITY;
    double den = 0.0, num = 0.0;
    for (int k = 0; k < D; ++k) {
        int t0, t1;
        float l0, l1;
        src_index<true>(sd, k, Dl, t0, t1, l0, l1);
        if (t0 != cur) {
            a0 = blend(t0);
            a1 = (t1 == t0) ? a0 : blend(t1);
            cur = t0;
        }
        const float v = l0 * a0 + l1 * a1;
        const float z = v * kNegLog2e;
        if (z > m) {
            const double f = (double)exp2f(m - z);  // m = -inf on the first bin -> 0
            den *= f;
            num *= f;
            m = z;
        }
        const float e = exp2f(z - m);
        den += (double)e;
        num += (double)e * (double)k;
    }
    const size_t o = (size_t)b * H * W + idx;
    disp[o] = (float)(num / den);
    if (stats) {
        stats[(size_t)b * 2 * H * W + idx] = m;
        stats[(size_t)b * 2 * H * W + (size_t)H * W + idx] = (float)(1.0 / den);
    }
}

}  // namespace rag
#include "disp_head_x3.cuh"
#include "disp_head_x3w.cuh"
#include "disp_head_x3r.cuh"
namespace rag {

// ---------------------------------------------------------------------------------------------
// generic backward: deterministic gather, one thread per low-res voxel.  Slow path / cross-check.
// ---------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT)
head_bwd_generic_kernel(const float* __restrict__ cost, const float* __restrict__ gdisp,
                        const float* __restrict__ disp, const float* __restrict__ stats,
                        float* __restrict__ gcost, int Dl, int Hl, int Wl, int D, float sd, float sh, float sw) {
    const int H = 3 * Hl, W = 3 * Wl;
    const size_t nvox = (size_t)Dl * Hl * Wl;
    const size_t idx = (size_t)blockIdx.x * NT + threadIdx.x;
    if (idx >= nvox) return;
    const int b = blockIdx.y;
    const int c = idx % Wl, r = (idx / Wl) % Hl, j = idx / ((size_t)Wl * Hl);
    const float* base = cost + (size_t)b * nvox;
    const size_t img = (size_t)H * W;
    const float* gd = gdisp + (size_t)b * img;
    const float* dp = disp + (size_t)b * img;
    const float* sm = stats + (size_t)b * 2 * img;
    const float* sinv = sm + img;

    // candidate full-res ranges (conservative), each candidate is tested against the tables
    const float inv_sd = 1.f / sd;
    const int klo = max(0, (int)floorf(((float)j - 0.5f) * inv_sd - 0.5f) - 2);
    const int khi = min(D - 1, (int)ceilf(((float)j + 1.5f) * inv_sd - 0.5f) + 2);
    const int hlo = max(0, 3 * r - 3), hhi = min(H - 1, 3 * r + 4);
    const int wlo = max(0, 3 * c - 3), whi = min(W - 1, 3 * c + 4);

    double acc = 0.0;
    for (int h = hlo; h <= hhi; ++h) {
        int h0, h1;
        float hl0, hl1;
        src_index<true>(sh, h, Hl, h0, h1, hl0, hl1);
        const float wh = (h0 == r ? hl0 : 0.f) + (h1 == r ? hl1 : 0.f);
        if (h0 != r && h1 != r) continue;
        for (int w = wlo; w <= whi; ++w) {
            int w0, w1;
            float wl0, wl1;
            src_index<true>(sw, w, Wl, w0, w1, wl0, wl1);
            if (w0 != c && w1 != c) continue;
            const float ww = (w0 == c ? wl0 : 0.f) + (w1 == c ? wl1 : 0.f);
            const size_t o = (size_t)h * W + w;
            const float g = __ldg(gd + o);
            if (g == 0.f) continue;
            const float dsp = __ldg(dp + o), m = __ldg(sm + o), inv = __ldg(sinv + o);
            const int o00 = h0 * Wl + w0, o01 = h0 * Wl + w1, o10 = h1 * Wl + w0, o11 = h1 * Wl + w1;
            auto blend = [&](int t) {
                const float* s = base + (size_t)t * Hl * Wl;
                return hl0 * (wl0 * __ldg(s + o00) + wl1 * __ldg(s + o01)) + hl1 * (wl0 * __ldg(s + o10) + wl1 * __ldg(s + o11));
            };
            double pix = 0.0;
            for (int k = klo; k <= khi; ++k) {
                int t0, t1;
                float l0, l1;
                src_index<true>(sd, k, Dl, t0, t1, l0, l1);
                if (t0 != j && t1 != j) continue;
                const float wd = (t0 == j ? l0 : 0.f) + (t1 == j ? l1 : 0.f);
                const float v = l0 * blend(t0) + l1 * blend(t1);
                const float p = exp2f(v * kNegLog2e - m) * inv;
                pix += (double)wd * (double)(-p * ((float)k - dsp));
            }
            acc += (double)(wh * ww) * (double)g * pix;
        }
    }
    gcost[(size_t)b * nvox + idx] = (float)acc;
}

// ---------------------------------------------------------------------------------------------
// DisparityRegression alone (rag_model.py:18-29) and its gradient
// ---------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT)
regression_fwd_kernel(const float* __restrict__ p, float* __restrict__ out, int D, int HW) {
    const int idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= HW) return;
    const int b = blockIdx.y;
    const float* s = p + (size_t)b * D * HW + idx;
    double acc = 0.0;
    int k = 0;
    for (; k + 4 <= D; k += 4) {
        const float v0 = ld_stream(s + (size_t)(k + 0) * HW), v1 = ld_stream(s + (size_t)(k + 1) * HW);
        const float v2 = ld_stream(s + (size_t)(k + 2) * HW), v3 = ld_stream(s + (size_t)(k + 3) * HW);
        acc += (double)v0 * k + (double)v1 * (k + 1) + (double)v2 * (k + 2) + (double)v3 * (k + 3);
    }
    for (; k < D; ++k) acc += (double)ld_stream(s + (size_t)k * HW) * k;
    out[(size_t)b * HW + idx] = (float)acc;
}

template <int NT>
__global__ void __launch_bounds__(NT)
regression_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gp, int D, int HW) {
    const int idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= HW) return;
    const int b = blockIdx.y;
    const float g = __ldg(gout + (size_t)b * HW + idx);
    float* d = gp + (size_t)b * D * HW + idx;
    for (int k = 0; k < D; ++k) st_stream(d + (size_t)k * HW, g * (float)k);
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static int check_head_args(int B, int Dl, int Hl, int Wl, int D) {
    if (B <= 0 || Dl <= 0 || Hl <= 0 || Wl <= 0 || D <= 0)
        return fail(RAG_E_SHAPE, "disp_head: non-positive dimension B=%d Dl=%d Hl=%d Wl=%d maxdisp=%d", B, Dl, Hl, Wl, D);
    if (B > 65535) return fail(RAG_E_SHAPE, "disp_head: B must be <= 65535");
    if ((size_t)9 * Hl * Wl >= ((size_t)1 << 31) || (size_t)Dl * Hl * Wl >= ((size_t)1 << 31) || D > 4096)
        return fail(RAG_E_SHAPE, "disp_head: image or volume too large (9*Hl*Wl, Dl*Hl*Wl < 2^31, maxdisp <= 4096)");
    return RAG_OK;
}

int upsample_trilinear(const float* cost, float* out, int B, int Dl, int Hl, int Wl, int D, int fma, cudaStream_t st) {
    if (!cost || !out) return fail(RAG_E_NULL, "upsample_trilinear: null pointer");
    if (int e = check_head_args(B, Dl, Hl, Wl, D)) return e;
    const size_t n = (size_t)D * 9 * Hl * Wl;
    const float sd = (float)Dl / (float)D, sh = (float)Hl / (float)(3 * Hl), sw = (float)Wl / (float)(3 * Wl);
    dim3 grid((unsigned)((n + 255) / 256), B);
    if (fma) upsample_kernel<true><<<grid, 256, 0, st>>>(cost, out, Dl, Hl, Wl, D, sd, sh, sw);
    else upsample_kernel<false><<<grid, 256, 0, st>>>(cost, out, Dl, Hl, Wl, D, sd, sh, sw);
    return check_launch("upsample_trilinear");
}

// variant: -1 = default; 0 = any (Dl, maxdisp) (one thread per output pixel, fp64 sums); 1 = first x3 kernel (any width);
// 2 = cube-root tiled kernel (default when maxdisp == 3*Dl, Wl % 4 == 0, 16-byte aligned input); 4 = RAG_HEAD_FWD_SHARED:
// variant 2 as a persistent grid of 3 CTAs per SM (SM sharing).  Id 3 (variant 2 with the lambda correction at every step
// and TwoSum totals) was retired: no default or schedule selected it.
int disp_head_fwd(const float* cost, float* disp, float* stats, int B, int Dl, int Hl, int Wl, int D,
                  int variant, cudaStream_t st) {
    if (!cost || !disp) return fail(RAG_E_NULL, "disp_head_fwd: null pointer");
    if (int e = check_head_args(B, Dl, Hl, Wl, D)) return e;
    if (variant < -1 || variant > 4 || variant == 3)
        return fail(RAG_E_VARIANT, "disp_head_fwd: unknown variant %d (id 3 was retired)", variant);
    const float sd = (float)Dl / (float)D, sh = (float)Hl / (float)(3 * Hl), sw = (float)Wl / (float)(3 * Wl);
    const bool x3 = (D == 3 * Dl);
    if (variant >= 1 && !x3) return fail(RAG_E_VARIANT, "disp_head_fwd: variant %d needs maxdisp == 3*Dl", variant);
    const bool persistent = variant == 4;      // RAG_HEAD_FWD_SHARED: variant 2 as a persistent grid of 3 CTAs per SM
    if (persistent) variant = 2;
    const bool tiled_ok = x3 && (Wl % 4 == 0) && aligned(cost, 16);
    if (variant >= 2 && !tiled_ok) return fail(RAG_E_VARIANT, "disp_head_fwd: variant %d needs maxdisp == 3*Dl, Wl %% 4 == 0 and 16-byte aligned cost_lr", variant);
    if (variant == -1) variant = tiled_ok ? 2 : (x3 ? 1 : 0);
    if (variant == 2) {
        // (5 block rows per CTA would fill the last wave of the 480x960 B=8 grid better, but 5 warps do not
        // spread evenly over the 4 SM sub-partitions: measured 202 us vs 165 us.)
        constexpr int warps = 4;
        const int nbx = (Wl + 31) / 32, nby = (Hl + warps - 1) / warps;
        const long long n_tl = (long long)nbx * nby * B;
        if (n_tl >= (1LL << 31)) return fail(RAG_E_SHAPE, "disp_head_fwd: too many tiles");
        const int grid = (int)(persistent ? std::min<long long>(n_tl, (long long)num_sms() * 3) : n_tl);
        const size_t smem = (size_t)2 * 16 * (warps + 2) * kTCols * sizeof(float) + ((size_t)18 * 32 * warps + 2 * Dl) * sizeof(float2);
        auto kern = head_fwd_x3r_kernel<warps, 4, 16, 2>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return fail((int)e, "disp_head_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        kern<<<grid, 32 * warps, smem, st>>>(cost, disp, stats, Dl, Hl, Wl, sd, nbx, nby, (int)n_tl);
    } else if (variant == 1) {
        constexpr int WARPS = 4;
        dim3 grid((Wl + 1 + 31) / 32, (Hl + 1 + WARPS - 1) / WARPS, B);
        head_fwd_x3_kernel<WARPS><<<grid, WARPS * 32, (size_t)D * sizeof(float), st>>>(cost, disp, stats, Dl, Hl, Wl, sd);
    } else {
        constexpr int NT = 128;
        dim3 grid((9 * Hl * Wl + NT - 1) / NT, B);
        head_fwd_generic_kernel<NT><<<grid, NT, 0, st>>>(cost, disp, stats, Dl, Hl, Wl, D, sd, sh, sw);
    }
    return check_launch("disp_head_fwd");
}

// variant: -1 = default; 0 = any-ratio gather; 1 = block-row tasks, one exp2 per pixel and k-block, both parts added
// in place with red.global.add (default when maxdisp == 3*Dl); 2 = same with the "B" part to `scratch` + a combine
// kernel (A/B; needs scratch); 3 = RAG_HEAD_BWD_SHARED: variant 1 as a persistent grid of 3 CTAs per SM (SM sharing)
int disp_head_bwd(const float* cost, const float* gdisp, const float* disp, const float* stats, float* gcost, float* scratch,
                  int B, int Dl, int Hl, int Wl, int D, int variant, cudaStream_t st) {
    if (!cost || !gdisp || !disp || !stats || !gcost) return fail(RAG_E_NULL, "disp_head_bwd: null pointer");
    if (int e = check_head_args(B, Dl, Hl, Wl, D)) return e;
    if (variant < -1 || variant > 3) return fail(RAG_E_VARIANT, "disp_head_bwd: unknown variant %d", variant);
    const float sd = (float)Dl / (float)D, sh = (float)Hl / (float)(3 * Hl), sw = (float)Wl / (float)(3 * Wl);
    const bool x3 = (D == 3 * Dl);
    if (variant >= 1 && !x3) return fail(RAG_E_VARIANT, "disp_head_bwd: variant %d needs maxdisp == 3*Dl", variant);
    if (variant == 2 && !scratch) return fail(RAG_E_NULL, "disp_head_bwd: variant 2 needs a scratch buffer");
    if (variant == -1) variant = x3 ? 1 : 0;
    if (variant >= 1) {
        const bool persistent = variant == 3;
        if (persistent) variant = 1;
        const int nJ = (Dl + kBwJ - 1) / kBwJ;
        const int strips = (Wl + 30) / 31;
        const int n_tasks = (Hl + 1) * nJ;
        const long long n_ct = (long long)strips * ((n_tasks + 3) / 4) * B;
        if (n_ct >= (1LL << 31)) return fail(RAG_E_SHAPE, "disp_head_bwd: too many tasks");
        const int grid = (int)(persistent ? std::min<long long>(n_ct, (long long)num_sms() * 3) : n_ct);
        const size_t smem = (size_t)3 * (D + 3) * sizeof(float2) + (size_t)4 * kBwWin * sizeof(float);
        auto kern = persistent ? head_bwd_x3w_kernel<true, true> : variant == 1 ? head_bwd_x3w_kernel<true> : head_bwd_x3w_kernel<false>;
        if (variant == 1) {   // two commutative contributions per element into a zeroed buffer (see the kernel's header)
            cudaError_t e = cudaMemsetAsync(gcost, 0, (size_t)B * Dl * Hl * Wl * sizeof(float), st);
            if (e != cudaSuccess) return fail((int)e, "disp_head_bwd: cudaMemsetAsync: %s", cudaGetErrorString(e));
        }
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return fail((int)e, "disp_head_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        }
        if (persistent) kern<<<grid, 128, smem, st>>>(cost, gdisp, disp, stats, gcost, scratch, Dl, Hl, Wl, sd, nJ, n_tasks, strips, (int)n_ct);
        else kern<<<dim3(strips, (n_tasks + 3) / 4, B), 128, smem, st>>>(cost, gdisp, disp, stats, gcost, scratch, Dl, Hl, Wl, sd, nJ, n_tasks, strips, (int)n_ct);
        if (int e = check_launch("disp_head_bwd(main)")) return e;
        if (variant == 1) return 0;
        const size_t n = (size_t)B * Dl * Hl * Wl;
        const size_t n4 = (aligned(gcost, 16) && aligned(scratch, 16)) ? n / 4 : 0;
        const size_t work = n4 > 0 ? n4 : 1;
        head_bwd_combine_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(gcost, scratch, n4, n);
        return check_launch("disp_head_bwd(combine)");
    }
    constexpr int NT = 128;
    const size_t nvox = (size_t)Dl * Hl * Wl;
    dim3 grid((unsigned)((nvox + NT - 1) / NT), B);
    head_bwd_generic_kernel<NT><<<grid, NT, 0, st>>>(cost, gdisp, disp, stats, gcost, Dl, Hl, Wl, D, sd, sh, sw);
    return check_launch("disp_head_bwd");
}

int disparity_regression_fwd(const float* p, float* out, int B, int D, int H, int W, cudaStream_t st) {
    if (!p || !out) return fail(RAG_E_NULL, "disparity_regression_fwd: null pointer");
    if (B <= 0 || D <= 0 || H <= 0 || W <= 0 || B > 65535 || (size_t)H * W >= ((size_t)1 << 31))
        return fail(RAG_E_SHAPE, "disparity_regression_fwd: bad shape B=%d D=%d H=%d W=%d", B, D, H, W);
    constexpr int NT = 256;
    dim3 grid((H * W + NT - 1) / NT, B);
    regression_fwd_kernel<NT><<<grid, NT, 0, st>>>(p, out, D, H * W);
    return check_launch("disparity_regression_fwd");
}

int disparity_regression_bwd(const float* gout, float* gp, int B, int D, int H, int W, cudaStream_t st) {
    if (!gout || !gp) return fail(RAG_E_NULL, "disparity_regression_bwd: null pointer");
    if (B <= 0 || D <= 0 || H <= 0 || W <= 0 || B > 65535 || (size_t)H * W >= ((size_t)1 << 31))
        return fail(RAG_E_SHAPE, "disparity_regression_bwd: bad shape B=%d D=%d H=%d W=%d", B, D, H, W);
    constexpr int NT = 256;
    dim3 grid((H * W + NT - 1) / NT, B);
    regression_bwd_kernel<NT><<<grid, NT, 0, st>>>(gout, gp, D, H * W);
    return check_launch("disparity_regression_bwd");
}

}  // namespace rag
