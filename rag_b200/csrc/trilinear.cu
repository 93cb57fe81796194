// Trilinear resize of a [B*C, Di, Hi, Wi] volume, forward and deterministic backward (SURVEY.md section 8f rank 2):
// the `upsample_6` / `upsample_12` branches of the Matching Net's tail, src/models/rag_model.py:356-366 and :675-685:
//     upsample_6  = nn.Upsample(size=x.size()[2:],        mode='trilinear', align_corners=True)
//     upsample_12 = nn.Upsample(size=[d//2, h//2, w//2],  mode='trilinear', align_corners=True)
// applied between last_12_3d / last_6_3d / last_3_3d, i.e. they produce the input of the layer that feeds the head.
//
// Arithmetic = PyTorch's (ATen/native/cuda/UpSample.cuh:96-130 + UpSampleTrilinear3d.cu), all fp32:
//     align_corners:  scale = (in-1)/(out-1) (0 if out == 1),  src = scale*dst
//     otherwise:      scale = in/out,                         src = max(scale*(dst+0.5)-0.5, 0)
//     i0 = (int)src, i1 = i0 + (i0 < in-1), l1 = src - i0, l0 = 1 - l1
//     out = t0*(h0*(w0*a000 + w1*a001) + h1*(w0*a010 + w1*a011)) + t1*(h0*(w0*a100 + w1*a101) + h1*(w0*a110 + w1*a111))
// Forward: one thread per 4 consecutive output columns (128-bit streaming stores; the input is 8x smaller and stays in
// L1/L2).  Backward: PyTorch scatters with atomicAdd (arrival order: not reproducible); here every INPUT voxel gathers the
// output voxels that reference it, in a fixed order -- the per-axis (i0, l1) tables and the first-destination index of
// every source index are built in shared memory by each CTA -- so the result is bitwise repeatable.
//
// Bilinear resize of a [B*C, Hi, Wi] image (rag_bilinear_resize_fwd/bwd: the cells' F.interpolate(..., 'bilinear')) runs the
// same kernels with the depth axis compiled out (template parameter D3 = false, Di = Do = 1): no depth weights, and an output
// row blends two input rows, not four.  A D = 1 view of the trilinear kernels would blend two copies of the same plane.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace rag {

template <bool AC>
__device__ __forceinline__ void tri_src(float scale, int dst, int n_in, int& i0, int& i1, float& l0, float& l1) {
    if (AC) {
        const float s = scale * (float)dst;
        i0 = min((int)s, n_in - 1);
        i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
        l1 = s - (float)i0;
        l0 = 1.f - l1;
    } else {
        src_index<true>(scale, dst, n_in, i0, i1, l0, l1);
    }
}

__host__ __device__ inline float tri_scale(int n_in, int n_out, bool ac) {
    if (ac) return n_out > 1 ? (float)(n_in - 1) / (float)(n_out - 1) : 0.f;
    return (float)n_in / (float)n_out;
}

// grid-stride over (bc, d, h, w-quad); Wo % 4 == 0 not required (scalar tail).
template <bool AC, bool D3>
__global__ void __launch_bounds__(256)
trilinear_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                     float sd, float sh, float sw, bool vec) {
    const int Wq = (Wo + 3) >> 2;
    const size_t n = (size_t)BC * Do * Ho * Wq;
    const size_t in_plane = (size_t)Hi * Wi, in_vol = (size_t)Di * in_plane;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        const int q = (int)(i % Wq);
        size_t r = i / Wq;
        const int h = (int)(r % Ho); r /= Ho;
        const int d = (int)(r % Do);
        const size_t bc = r / Do;
        int d0 = 0, d1 = 0, h0, h1;
        float t0, t1, e0, e1;
        if constexpr (D3) tri_src<AC>(sd, d, Di, d0, d1, t0, t1);
        tri_src<AC>(sh, h, Hi, h0, h1, e0, e1);
        const float* p = in + bc * in_vol;
        const float* r00 = p + (size_t)d0 * in_plane + (size_t)h0 * Wi;
        const float* r01 = p + (size_t)d0 * in_plane + (size_t)h1 * Wi;
        const float* r10 = p + (size_t)d1 * in_plane + (size_t)h0 * Wi;
        const float* r11 = p + (size_t)d1 * in_plane + (size_t)h1 * Wi;
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int w = 4 * q + k;
            int w0, w1;
            float f0, f1;
            tri_src<AC>(sw, min(w, Wo - 1), Wi, w0, w1, f0, f1);
            if constexpr (D3)
                v[k] = t0 * (e0 * (f0 * __ldg(r00 + w0) + f1 * __ldg(r00 + w1)) + e1 * (f0 * __ldg(r01 + w0) + f1 * __ldg(r01 + w1))) +
                       t1 * (e0 * (f0 * __ldg(r10 + w0) + f1 * __ldg(r10 + w1)) + e1 * (f0 * __ldg(r11 + w0) + f1 * __ldg(r11 + w1)));
            else
                v[k] = e0 * (f0 * __ldg(r00 + w0) + f1 * __ldg(r00 + w1)) + e1 * (f0 * __ldg(r01 + w0) + f1 * __ldg(r01 + w1));
        }
        float* o = out + ((bc * Do + d) * Ho + h) * (size_t)Wo + 4 * q;
        if (vec) {
            st_stream(reinterpret_cast<float4*>(o), make_float4(v[0], v[1], v[2], v[3]));
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * q + k < Wo) o[k] = v[k];
        }
    }
}

// Per-axis tables in shared memory: i0[dst], l1[dst] for dst < n_out and first[i] = smallest dst with i0[dst] >= i for i <= n_in.
template <bool AC>
__device__ void tri_tables(float scale, int n_in, int n_out, int* i0t, float* l1t, int* first) {
    for (int dst = threadIdx.x; dst < n_out; dst += blockDim.x) {
        int a, b;
        float l0, l1;
        tri_src<AC>(scale, dst, n_in, a, b, l0, l1);
        i0t[dst] = a;
        l1t[dst] = l1;
    }
    __syncthreads();
    for (int dst = threadIdx.x; dst <= n_out; dst += blockDim.x) {
        const int prev = dst == 0 ? -1 : i0t[dst - 1];
        const int cur = dst == n_out ? n_in : i0t[dst];      // sentinel: every remaining source index starts past the end
        for (int i = prev + 1; i <= cur; ++i) first[i] = dst;
    }
    __syncthreads();
}

// gin[bc, id, ih, iw] = sum over the output voxels that read it of (weight * gout).  One thread per input voxel.
// smem: per axis  int i0[n_out] | float l1[n_out] | int first[n_in + 1]
template <bool AC, bool D3>
__global__ void __launch_bounds__(256)
trilinear_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                     float sd, float sh, float sw) {
    extern __shared__ int tri_smem[];
    int* d_i0 = tri_smem;            float* d_l1 = reinterpret_cast<float*>(d_i0 + Do); int* d_first = reinterpret_cast<int*>(d_l1 + Do);
    int* h_i0 = d_first + Di + 1;    float* h_l1 = reinterpret_cast<float*>(h_i0 + Ho); int* h_first = reinterpret_cast<int*>(h_l1 + Ho);
    int* w_i0 = h_first + Hi + 1;    float* w_l1 = reinterpret_cast<float*>(w_i0 + Wo); int* w_first = reinterpret_cast<int*>(w_l1 + Wo);
    if constexpr (D3) tri_tables<AC>(sd, Di, Do, d_i0, d_l1, d_first);
    tri_tables<AC>(sh, Hi, Ho, h_i0, h_l1, h_first);
    tri_tables<AC>(sw, Wi, Wo, w_i0, w_l1, w_first);
    const size_t n = (size_t)BC * Di * Hi * Wi;
    const size_t out_plane = (size_t)Ho * Wo, out_vol = (size_t)Do * out_plane;
    // weight of destination `dst` on source index i along an axis with tables (i0, l1), n_in sources
    auto wgt = [](int i, int a, float l1, int n_in) -> float {
        const int b = a + (a < n_in - 1 ? 1 : 0);
        return (a == i ? 1.f - l1 : 0.f) + (b == i ? l1 : 0.f);
    };
    for (size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x; idx < n; idx += (size_t)gridDim.x * 256) {
        const int iw = (int)(idx % Wi);
        size_t r = idx / Wi;
        const int ih = (int)(r % Hi); r /= Hi;
        const int id = (int)(r % Di);
        const size_t bc = r / Di;
        int dl = 0, dh = 1;                                                 // 2-D: the one plane, weight 1
        if constexpr (D3) dl = d_first[max(id - 1, 0)], dh = d_first[id + 1];   // destinations with i0 in {id-1, id}
        const int hl = h_first[max(ih - 1, 0)], hh = h_first[ih + 1];
        const int wl = w_first[max(iw - 1, 0)], wh = w_first[iw + 1];
        const float* gp = gout + bc * out_vol;
        float acc = 0.f;
        if (wh - wl <= 5) {
            // common case (up-sampling by ~2-3): at most five destinations per axis.  The w weights live in registers and
            // the five loads per row are unconditional (clamped column, zero weight) -- no table look-ups in the inner loop.
            float ww[5];
            int wc[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const int w = wl + k;
                wc[k] = min(w, Wo - 1);
                ww[k] = w < wh ? wgt(iw, w_i0[wc[k]], w_l1[wc[k]], Wi) : 0.f;
            }
            for (int d = dl; d < dh; ++d) {
                const float wd = D3 ? wgt(id, d_i0[d], d_l1[d], Di) : 1.f;
                float accd = 0.f;
                for (int h = hl; h < hh; ++h) {
                    const float whh = wgt(ih, h_i0[h], h_l1[h], Hi);
                    const float* row = gp + (size_t)d * out_plane + (size_t)h * Wo;
                    float acch = ww[0] * __ldg(row + wc[0]);
#pragma unroll
                    for (int k = 1; k < 5; ++k) acch = __fmaf_rn(ww[k], __ldg(row + wc[k]), acch);
                    accd = __fmaf_rn(whh, acch, accd);
                }
                acc = __fmaf_rn(wd, accd, acc);
            }
        } else {
            for (int d = dl; d < dh; ++d) {
                const float wd = D3 ? wgt(id, d_i0[d], d_l1[d], Di) : 1.f;
                if (wd == 0.f) continue;
                float accd = 0.f;
                for (int h = hl; h < hh; ++h) {
                    const float whh = wgt(ih, h_i0[h], h_l1[h], Hi);
                    if (whh == 0.f) continue;
                    const float* row = gp + (size_t)d * out_plane + (size_t)h * Wo;
                    float acch = 0.f;
                    for (int w = wl; w < wh; ++w) acch = __fmaf_rn(wgt(iw, w_i0[w], w_l1[w], Wi), __ldg(row + w), acch);
                    accd = __fmaf_rn(whh, acch, accd);
                }
                acc = __fmaf_rn(wd, accd, acc);
            }
        }
        gin[idx] = acc;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Row kernels (default for the network's shapes: Wi % 4 == 0, Wo % 4 == 0, at most five destinations per source column).
// The kernels above spend ~37 instructions per output (32 scalar loads + four source-index evaluations per thread) and
// up to 125 loads per input voxel: 0.19 + 0.37 ms at [4,12,32,48,96] -> [4,12,64,96,192] against an HBM floor of
// 0.036 ms each.  The interpolation is separable, so here a WARP owns a row:
//   forward   the four input rows an output row interpolates between are blended into ONE row of Wi values (128-bit
//             loads, shared memory), then every lane interpolates its output columns from that row -- the (i0, l1) of a
//             lane's columns are the same for every row and live in registers;
//   backward  the (at most 5 x 5) output rows that reference an input row are combined with their depth x height weights
//             into ONE row of Wo values (128-bit loads), then every lane gathers its input columns from it with the
//             column weights it keeps in registers.  Every sum runs in a fixed order: bitwise repeatable.
// The order of the roundings differs from ATen's (depth/height first instead of width first): 1e-7 relative.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kTriWarps = 8;
constexpr int kTriList = 32;              // output rows per input row the backward row kernel lists at a time (5 x 5 fit)

// grid-stride over output rows; smem: float [kTriWarps][Wi + 4]
// NPER / NVI = 128-bit vectors per lane of an output row (ceil(Wo / 128)) / of an input row; PF: fetch the input rows one
// output row ahead (pays for wide rows -- 0.73 -> 0.54 ms at [8,12,32,80,160] -> [64,160,320] --, costs at narrow ones:
// 0.093 -> 0.108 ms at [4,12,32,48,96] -> [64,96,192])
template <bool AC, int NPER, int NVI, bool PF, bool D3>
__global__ void __launch_bounds__(kTriWarps * 32)
trilinear_fwd_rows_kernel(const float* __restrict__ in, float* __restrict__ out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                          float sd, float sh, float sw) {
    extern __shared__ __align__(16) float tri_rows[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* rb = tri_rows + warp * (Wi + 4);
    const int Wiv = Wi >> 2, Wov = Wo >> 2;
    // the lane's output columns: where they read the blended row and both weights, once
    const float* cp[NPER][4];
    float cl0[NPER][4], cl[NPER][4];
#pragma unroll
    for (int p = 0; p < NPER; ++p)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int w = min(4 * (lane + 32 * p) + k, Wo - 1);
            int i0, i1;
            tri_src<AC>(sw, w, Wi, i0, i1, cl0[p][k], cl[p][k]);
            cp[p][k] = rb + i0;
        }
    const size_t in_plane = (size_t)Hi * Wi, in_vol = (size_t)Di * in_plane;
    const long long n_rows = (long long)BC * Do * Ho;
    const long long stride = (long long)gridDim.x * kTriWarps;
    // the four input rows of an output row (NVI vectors per lane) and its depth / height weights: fetched
    // one row AHEAD, so the loads of row k+1 are in flight while row k is blended, interpolated and stored
    struct RowCtx {
        float4 a[NVI], b[NVI], c[NVI], e[NVI];
        float t0, t1, e0, e1;
    };
    // the row index advances by `stride` rows, i.e. by fixed digits in the mixed radix (Ho, Do, BC): no division per row
    const int sq = (int)(stride / Ho), inc_h = (int)(stride - (long long)sq * Ho);
    const int inc_bc = sq / Do, inc_d = sq - inc_bc * Do;
    int f_h, f_d, f_bc;                            // digits of the next row to FETCH
    {
        const long long r0 = (long long)blockIdx.x * kTriWarps + warp;
        f_h = (int)(r0 % Ho);
        f_d = (int)((r0 / Ho) % Do);
        f_bc = (int)(r0 / ((long long)Ho * Do));
    }
    auto fetch = [&](RowCtx& r) {                  // fetches row (f_bc, f_d, f_h) and advances the digits
        const int h = f_h, d = f_d;
        const size_t bc = (size_t)f_bc;
        f_h += inc_h; if (f_h >= Ho) { f_h -= Ho; ++f_d; }
        f_d += inc_d; if (f_d >= Do) { f_d -= Do; ++f_bc; }
        f_bc += inc_bc;
        int d0 = 0, d1 = 0, h0, h1;
        if constexpr (D3) tri_src<AC>(sd, d, Di, d0, d1, r.t0, r.t1);
        tri_src<AC>(sh, h, Hi, h0, h1, r.e0, r.e1);
        const float* p = in + bc * in_vol;
        const float4* r00 = reinterpret_cast<const float4*>(p + (size_t)d0 * in_plane + (size_t)h0 * Wi);
        const float4* r01 = reinterpret_cast<const float4*>(p + (size_t)d0 * in_plane + (size_t)h1 * Wi);
        const float4* r10 = reinterpret_cast<const float4*>(p + (size_t)d1 * in_plane + (size_t)h0 * Wi);
        const float4* r11 = reinterpret_cast<const float4*>(p + (size_t)d1 * in_plane + (size_t)h1 * Wi);
#pragma unroll
        for (int j = 0; j < NVI; ++j) {
            const int v = lane + 32 * j;
            if (v < Wiv) {
                r.a[j] = __ldg(r00 + v); r.b[j] = __ldg(r01 + v);
                if constexpr (D3) { r.c[j] = __ldg(r10 + v); r.e[j] = __ldg(r11 + v); }
            }
        }
    };
    long long row = (long long)blockIdx.x * kTriWarps + warp;
    RowCtx cur, nxt;
    if (PF && row < n_rows) fetch(cur);
    for (; row < n_rows; row += stride) {
        if (PF) {
            if (row + stride < n_rows) fetch(nxt);
        } else {
            fetch(cur);
        }
        __syncwarp();                              // the previous row's reads of rb are done
#pragma unroll
        for (int j = 0; j < NVI; ++j) {
            const int v = lane + 32 * j;
            if (v < Wiv) {
                const float4 a = cur.a[j], b = cur.b[j], c = cur.c[j], e = cur.e[j];
                const float t0 = cur.t0, t1 = cur.t1, e0 = cur.e0, e1 = cur.e1;
                float4 o;
                if constexpr (D3) {
                    o.x = t0 * (e0 * a.x + e1 * b.x) + t1 * (e0 * c.x + e1 * e.x);
                    o.y = t0 * (e0 * a.y + e1 * b.y) + t1 * (e0 * c.y + e1 * e.y);
                    o.z = t0 * (e0 * a.z + e1 * b.z) + t1 * (e0 * c.z + e1 * e.z);
                    o.w = t0 * (e0 * a.w + e1 * b.w) + t1 * (e0 * c.w + e1 * e.w);
                } else {
                    o.x = e0 * a.x + e1 * b.x; o.y = e0 * a.y + e1 * b.y; o.z = e0 * a.z + e1 * b.z; o.w = e0 * a.w + e1 * b.w;
                }
                reinterpret_cast<float4*>(rb)[v] = o;
                if (v == Wiv - 1) rb[Wi] = o.w;   // "i0 + 1" of the last source column is the column itself (i1 == i0 there)
            }
        }
        __syncwarp();
        float4* o4 = reinterpret_cast<float4*>(out + (size_t)row * Wo);
#pragma unroll
        for (int pp = 0; pp < NPER; ++pp) {
            const int q = lane + 32 * pp;
            if (q < Wov) {
                float v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = cl0[pp][k] * cp[pp][k][0] + cl[pp][k] * cp[pp][k][1];
                st_stream(o4 + q, make_float4(v[0], v[1], v[2], v[3]));
            }
        }
        if (PF) cur = nxt;
    }
}

// grid-stride over input rows; smem: the three axes' tables (as trilinear_bwd_kernel) | int wfirst[Wi] | float wk[5][Wi]
// (per source column: its first destination and the weights of the five destinations from there on, 0 past the last) |
// float [kTriWarps][Wo + 4]
template <bool AC, int NPER, bool D3>   // NPER = 128-bit vectors of an output row per lane
__global__ void __launch_bounds__(kTriWarps * 32)
trilinear_bwd_rows_kernel(const float* __restrict__ gout, float* __restrict__ gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                          float sd, float sh, float sw) {
    extern __shared__ __align__(16) int tri_smem2[];
    int* d_i0 = tri_smem2;           float* d_l1 = reinterpret_cast<float*>(d_i0 + Do); int* d_first = reinterpret_cast<int*>(d_l1 + Do);
    int* h_i0 = d_first + Di + 1;    float* h_l1 = reinterpret_cast<float*>(h_i0 + Ho); int* h_first = reinterpret_cast<int*>(h_l1 + Ho);
    int* w_i0 = h_first + Hi + 1;    float* w_l1 = reinterpret_cast<float*>(w_i0 + Wo); int* w_first = reinterpret_cast<int*>(w_l1 + Wo);
    int* wfirst = w_first + Wi + 1;
    float* wk = reinterpret_cast<float*>(wfirst + Wi);
    float* rows = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(wk + 5 * Wi) + 15) & ~(uintptr_t)15);
    // per warp: the output rows that reference the current input row as a flat list (row offset in vectors, depth x height weight)
    int* lst_off = reinterpret_cast<int*>(rows + kTriWarps * (Wo + 4)) + (threadIdx.x >> 5) * kTriList;
    float* lst_w = reinterpret_cast<float*>(reinterpret_cast<int*>(rows + kTriWarps * (Wo + 4)) + kTriWarps * kTriList) + (threadIdx.x >> 5) * kTriList;
    if constexpr (D3) tri_tables<AC>(sd, Di, Do, d_i0, d_l1, d_first);
    tri_tables<AC>(sh, Hi, Ho, h_i0, h_l1, h_first);
    tri_tables<AC>(sw, Wi, Wo, w_i0, w_l1, w_first);
    auto wgt = [](int i, int a, float l1, int n_in) -> float {
        const int b = a + (a < n_in - 1 ? 1 : 0);
        return (a == i ? 1.f - l1 : 0.f) + (b == i ? l1 : 0.f);
    };
    for (int iw = threadIdx.x; iw < Wi; iw += blockDim.x) {
        const int wl = w_first[max(iw - 1, 0)], wh = w_first[iw + 1];
        wfirst[iw] = wl;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int w = wl + k, wc = min(w, Wo - 1);
            wk[k * Wi + iw] = w < wh ? wgt(iw, w_i0[wc], w_l1[wc], Wi) : 0.f;
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* tmp = rows + warp * (Wo + 4);
    const int Wov = Wo >> 2;
    const size_t out_plane = (size_t)Ho * Wo, out_vol = (size_t)Do * out_plane;
    const long long n_rows = (long long)BC * Di * Hi;
    // the row index advances by fixed digits in the mixed radix (Hi, Di, BC): no division per row
    const long long stride = (long long)gridDim.x * kTriWarps;
    const int sq = (int)(stride / Hi), inc_h = (int)(stride - (long long)sq * Hi);
    const int inc_bc = sq / Di, inc_d = sq - inc_bc * Di;
    long long row = (long long)blockIdx.x * kTriWarps + warp;
    int ih = (int)(row % Hi), id = (int)((row / Hi) % Di), ibc = (int)(row / ((long long)Hi * Di));
    for (; row < n_rows; row += stride) {
        const size_t bc = (size_t)ibc;
        int dl = 0, dh = 1;                                                 // 2-D: the one plane, weight 1
        if constexpr (D3) dl = d_first[max(id - 1, 0)], dh = d_first[id + 1];   // destinations with i0 in {id-1, id}
        const int hl = h_first[max(ih - 1, 0)], hh = h_first[ih + 1];
        const float* gp = gout + bc * out_vol;
        const int c_id = id, c_ih = ih;
        ih += inc_h; if (ih >= Hi) { ih -= Hi; ++id; }
        id += inc_d; if (id >= Di) { id -= Di; ++ibc; }
        ibc += inc_bc;
        float4 acc[NPER];
#pragma unroll
        for (int pp = 0; pp < NPER; ++pp) acc[pp] = make_float4(0.f, 0.f, 0.f, 0.f);
        // The (dh - dl) x (hh - hl) referencing output rows as ONE flat list in shared memory -- a lane computes one entry
        // (row offset, depth x height weight) --, walked two or four entries at a time with all their loads issued first: the
        // nested loops recomputed the height weight for every depth and exposed one L2 round trip per output row.
        const int nh = hh - hl, n_ref = (dh - dl) * nh;
        for (int base = 0; base < n_ref; base += kTriList) {
            const int n_here = min(kTriList, n_ref - base);
            __syncwarp();
            if (lane < n_here) {
                const int e = base + lane, dd = e / nh, d = dl + dd, h = hl + (e - dd * nh);
                lst_off[lane] = (int)(((size_t)d * out_plane + (size_t)h * Wo) >> 2);
                if constexpr (D3) lst_w[lane] = wgt(c_id, d_i0[d], d_l1[d], Di) * wgt(c_ih, h_i0[h], h_l1[h], Hi);
                else lst_w[lane] = wgt(c_ih, h_i0[h], h_l1[h], Hi);
            }
            __syncwarp();
            const float4* g4 = reinterpret_cast<const float4*>(gp) + lane;
            constexpr int U = NPER >= 3 ? 2 : 4;   // entries in flight: 8 vectors per lane at most (more costs occupancy)
            int e = 0;
            for (; e + U <= n_here; e += U) {
                float4 g[U][NPER];
                float c[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    c[u] = lst_w[e + u];
                    const float4* r4 = g4 + lst_off[e + u];
#pragma unroll
                    for (int pp = 0; pp < NPER; ++pp)
                        g[u][pp] = lane + 32 * pp < Wov ? ld_stream(r4 + 32 * pp) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int pp = 0; pp < NPER; ++pp) {
                        acc[pp].x = __fmaf_rn(c[u], g[u][pp].x, acc[pp].x); acc[pp].y = __fmaf_rn(c[u], g[u][pp].y, acc[pp].y);
                        acc[pp].z = __fmaf_rn(c[u], g[u][pp].z, acc[pp].z); acc[pp].w = __fmaf_rn(c[u], g[u][pp].w, acc[pp].w);
                    }
            }
            for (; e < n_here; ++e) {
                const float c = lst_w[e];
                const float4* r4 = g4 + lst_off[e];
#pragma unroll
                for (int pp = 0; pp < NPER; ++pp) {
                    if (lane + 32 * pp < Wov) {
                        const float4 g = ld_stream(r4 + 32 * pp);
                        acc[pp].x = __fmaf_rn(c, g.x, acc[pp].x); acc[pp].y = __fmaf_rn(c, g.y, acc[pp].y);
                        acc[pp].z = __fmaf_rn(c, g.z, acc[pp].z); acc[pp].w = __fmaf_rn(c, g.w, acc[pp].w);
                    }
                }
            }
        }
        __syncwarp();                              // the previous row's gathers from tmp are done
#pragma unroll
        for (int pp = 0; pp < NPER; ++pp) {
            const int q = lane + 32 * pp;
            if (q < Wov) reinterpret_cast<float4*>(tmp)[q] = acc[pp];
        }
        __syncwarp();
        float* go = gin + (size_t)row * Wi;
        for (int iw = lane; iw < Wi; iw += 32) {
            const int wl = wfirst[iw];
            float a = wk[iw] * tmp[min(wl, Wo - 1)];
#pragma unroll
            for (int k = 1; k < 5; ++k) a = __fmaf_rn(wk[k * Wi + iw], tmp[min(wl + k, Wo - 1)], a);
            go[iw] = a;
        }
    }
}

// largest number of destinations that reference one source index (i0 in {i-1, i}) along an axis, evaluated on the host with
// the kernel's own fp32 arithmetic
static int tri_max_refs(int n_in, int n_out, bool ac) {
    const float scale = tri_scale(n_in, n_out, ac);
    std::vector<int> i0(n_out);
    for (int dst = 0; dst < n_out; ++dst) {
        float s = ac ? scale * (float)dst : fmaf(scale, (float)dst + 0.5f, -0.5f);
        if (!ac && s < 0.f) s = 0.f;
        i0[dst] = ac ? std::min((int)s, n_in - 1) : (int)s;
    }
    std::vector<int> cnt(n_in + 1, 0);
    for (int dst = 0; dst < n_out; ++dst) {
        cnt[i0[dst]]++;
        if (i0[dst] + 1 < n_in) cnt[i0[dst] + 1]++;
    }
    return *std::max_element(cnt.begin(), cnt.end());
}

static int check_tri(const char* who, const void* a, const void* b, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo) {
    if (!a || !b) return fail(RAG_E_NULL, "%s: null pointer", who);
    if (BC <= 0 || Di <= 0 || Hi <= 0 || Wi <= 0 || Do <= 0 || Ho <= 0 || Wo <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    if ((size_t)Di * Hi * Wi >= ((size_t)1 << 31) || (size_t)Do * Ho * Wo >= ((size_t)1 << 31))
        return fail(RAG_E_SHAPE, "%s: a volume must have fewer than 2^31 voxels", who);
    if ((size_t)(Do + Ho + Wo) * 8 + (size_t)(Di + Hi + Wi + 3) * 4 > 160 * 1024) return fail(RAG_E_SHAPE, "%s: axes too long for the shared-memory tables", who);
    if (!aligned(a, 4) || !aligned(b, 4)) return fail(RAG_E_ALIGN, "%s: pointers must be 4-byte aligned", who);
    return RAG_OK;
}

// D3 = false: the bilinear exports (Di = Do = 1, depth compiled out); `who` names the export in errors
template <bool D3>
static int resize_fwd(const char* who, const float* in, float* out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners,
                      cudaStream_t st) {
    if (int e = check_tri(who, in, out, BC, Di, Hi, Wi, Do, Ho, Wo)) return e;
    const bool ac = align_corners != 0;
    const float sd = tri_scale(Di, Do, ac), sh = tri_scale(Hi, Ho, ac), sw = tri_scale(Wi, Wo, ac);
    // row kernel: 128-bit rows on both sides, an input row within 2 and an output row within 4 vectors per lane
    if (Wi % 4 == 0 && Wi <= 256 && Wo % 4 == 0 && Wo <= 512 && aligned(in, 16) && aligned(out, 16)) {
        const int nper = (Wo / 4 + 31) / 32;
        const size_t smem = (size_t)kTriWarps * (Wi + 4) * sizeof(float);
        const long long n_rows = (long long)BC * Do * Ho;
        const unsigned grid = (unsigned)std::min<long long>((n_rows + kTriWarps - 1) / kTriWarps, (long long)num_sms() * 16);
        auto launch = [&](auto kern) -> int {
            if (smem > 48 * 1024) {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));
            }
            kern<<<grid, kTriWarps * 32, smem, st>>>(in, out, BC, Di, Hi, Wi, Do, Ho, Wo, sd, sh, sw);
            return RAG_OK;
        };
        int rc = RAG_OK;
        if (smem <= 160 * 1024) {
#define RAG_TRI_FWD(ACV, NV)                                                                                              \
    (nper == 1 ? launch(trilinear_fwd_rows_kernel<ACV, 1, NV, (NV > 1), D3>) : nper == 2 ? launch(trilinear_fwd_rows_kernel<ACV, 2, NV, (NV > 1), D3>) \
     : nper == 3 ? launch(trilinear_fwd_rows_kernel<ACV, 3, NV, (NV > 1), D3>) : launch(trilinear_fwd_rows_kernel<ACV, 4, NV, (NV > 1), D3>))
            // wider input rows (the cells' level-3 rows: 320 at 480x960, 416 at 384x1248) stay on the per-voxel kernel: row
            // kernels with 3 and 4 input vectors per lane were measured no faster there (DESIGN.md 5.12)
            const bool one = Wi <= 128;
            rc = ac ? (one ? RAG_TRI_FWD(true, 1) : RAG_TRI_FWD(true, 2)) : (one ? RAG_TRI_FWD(false, 1) : RAG_TRI_FWD(false, 2));
#undef RAG_TRI_FWD
            if (rc) return rc;
            return check_launch(D3 ? "trilinear_resize_fwd(rows)" : "bilinear_resize_fwd(rows)");
        }
    }
    const size_t n = (size_t)BC * Do * Ho * ((Wo + 3) / 4);
    const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)num_sms() * 32);
    const bool vec = Wo % 4 == 0 && aligned(out, 16);
    if (ac) trilinear_fwd_kernel<true, D3><<<grid, 256, 0, st>>>(in, out, BC, Di, Hi, Wi, Do, Ho, Wo, sd, sh, sw, vec);
    else trilinear_fwd_kernel<false, D3><<<grid, 256, 0, st>>>(in, out, BC, Di, Hi, Wi, Do, Ho, Wo, sd, sh, sw, vec);
    return check_launch(who);
}

template <bool D3>
static int resize_bwd(const char* who, const float* gout, float* gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners,
                      cudaStream_t st) {
    if (int e = check_tri(who, gout, gin, BC, Di, Hi, Wi, Do, Ho, Wo)) return e;
    const bool ac = align_corners != 0;
    const float sd = tri_scale(Di, Do, ac), sh = tri_scale(Hi, Ho, ac), sw = tri_scale(Wi, Wo, ac);
    const size_t smem = (size_t)(Do + Ho + Wo) * 8 + (size_t)(Di + Hi + Wi + 3) * 4;
    // row kernel: 128-bit output rows of at most 4 vectors per lane, at most five destinations per source column (any
    // up-sampling by a factor <= 2)
    if (Wo % 4 == 0 && Wo <= 512 && aligned(gout, 16) && tri_max_refs(Wi, Wo, ac) <= 5) {
        const int nper = (Wo / 4 + 31) / 32;
        const size_t smem2 = smem + (size_t)6 * Wi * 4 + 16 + (size_t)kTriWarps * (Wo + 4) * sizeof(float) + (size_t)kTriWarps * kTriList * 8;
        const long long n_rows = (long long)BC * Di * Hi;
        const unsigned grid = (unsigned)std::min<long long>((n_rows + kTriWarps - 1) / kTriWarps, (long long)num_sms() * 8);
        auto launch = [&](auto kern) -> int {
            if (smem2 > 48 * 1024) {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
                if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));
            }
            kern<<<grid, kTriWarps * 32, smem2, st>>>(gout, gin, BC, Di, Hi, Wi, Do, Ho, Wo, sd, sh, sw);
            return RAG_OK;
        };
        if (smem2 <= 160 * 1024) {
            int rc;
            if (ac) rc = nper == 1 ? launch(trilinear_bwd_rows_kernel<true, 1, D3>) : nper == 2 ? launch(trilinear_bwd_rows_kernel<true, 2, D3>) : nper == 3 ? launch(trilinear_bwd_rows_kernel<true, 3, D3>) : launch(trilinear_bwd_rows_kernel<true, 4, D3>);
            else rc = nper == 1 ? launch(trilinear_bwd_rows_kernel<false, 1, D3>) : nper == 2 ? launch(trilinear_bwd_rows_kernel<false, 2, D3>) : nper == 3 ? launch(trilinear_bwd_rows_kernel<false, 3, D3>) : launch(trilinear_bwd_rows_kernel<false, 4, D3>);
            if (rc) return rc;
            return check_launch(D3 ? "trilinear_resize_bwd(rows)" : "bilinear_resize_bwd(rows)");
        }
    }
    const size_t n = (size_t)BC * Di * Hi * Wi;
    const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)num_sms() * 16);
    auto kern = ac ? trilinear_bwd_kernel<true, D3> : trilinear_bwd_kernel<false, D3>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));
    }
    kern<<<grid, 256, smem, st>>>(gout, gin, BC, Di, Hi, Wi, Do, Ho, Wo, sd, sh, sw);
    return check_launch(who);
}

int trilinear_resize_fwd(const float* in, float* out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners, cudaStream_t st) {
    return resize_fwd<true>("trilinear_resize_fwd", in, out, BC, Di, Hi, Wi, Do, Ho, Wo, align_corners, st);
}

int trilinear_resize_bwd(const float* gout, float* gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners, cudaStream_t st) {
    return resize_bwd<true>("trilinear_resize_bwd", gout, gin, BC, Di, Hi, Wi, Do, Ho, Wo, align_corners, st);
}

int bilinear_resize_fwd(const float* in, float* out, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners, cudaStream_t st) {
    return resize_fwd<false>("bilinear_resize_fwd", in, out, BC, 1, Hi, Wi, 1, Ho, Wo, align_corners, st);
}

int bilinear_resize_bwd(const float* gout, float* gin, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners, cudaStream_t st) {
    return resize_bwd<false>("bilinear_resize_bwd", gout, gin, BC, 1, Hi, Wi, 1, Ho, Wo, align_corners, st);
}

}  // namespace rag
