// Concatenation cost volume, forward and backward, for sm_100a.
//
// Reference semantics: src/models/rag_model.py:375-383 (and its two verbatim copies):
//   cost[b,   c, d,h,w] = x[b,c,h,w]   (w >= d) else 0
//   cost[b, C+c, d,h,w] = y[b,c,h,w-d] (w >= d) else 0
// The reference does this with one zero-fill + 2*Df strided slice copies (129 launches, the
// volume written twice) and its autograd replays 2*Df CopySlices nodes that each clone the full
// gradient volume.  Here: one launch per direction, every byte of the volume touched once.
//
// Forward  (HBM store stream): a CTA stages R feature rows of one (b,c) -- the left row once and
//   the right row as V copies pre-shifted by 0..V-1 elements -- in shared memory, so that for every
//   disparity d = V*q + s the shifted right row is an ALIGNED 16-byte shared-memory read of copy s
//   at vector offset -q, and every global store is a full, aligned, coalesced 128-bit store.
//   Each input row is read from HBM/L2 once per disparity sweep (d-chunk), not once per disparity.
// Backward (HBM load stream): one thread owns V adjacent w of one (b,c,h) row and walks d from
//   Df-1 down to 0 accumulating in fp32 -- exactly the order in which autograd accumulates the
//   CopySlices gradients -- so the result is bit-identical to the reference; loads are 128-bit,
//   coalesced, and issued U disparities ahead of the dependent adds.  No atomics, no reduction tree.
#include <cuda_pipeline.h>

#include <algorithm>

#include "common.cuh"
#include "cv_lean.cuh"

namespace rag {

template <int V> struct Vec;
template <> struct Vec<4> { using T = float4; };
template <> struct Vec<2> { using T = float2; };
template <> struct Vec<1> { using T = float; };

__device__ __forceinline__ float get(const float4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
__device__ __forceinline__ float get(const float2& v, int i) { return i == 0 ? v.x : v.y; }
__device__ __forceinline__ float get(const float& v, int) { return v; }
__device__ __forceinline__ void set(float4& v, int i, float a) { if (i == 0) v.x = a; else if (i == 1) v.y = a; else if (i == 2) v.z = a; else v.w = a; }
__device__ __forceinline__ void set(float2& v, int i, float a) { if (i == 0) v.x = a; else v.y = a; }
__device__ __forceinline__ void set(float& v, int, float a) { v = a; }
template <typename T> __device__ __forceinline__ T zero_vec();
template <> __device__ __forceinline__ float4 zero_vec<float4>() { return make_float4(0.f, 0.f, 0.f, 0.f); }
template <> __device__ __forceinline__ float2 zero_vec<float2>() { return make_float2(0.f, 0.f); }
template <> __device__ __forceinline__ float zero_vec<float>() { return 0.f; }

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// One work unit = R rows of one (b,c) x one sweep of `dchunk` disparities.
// smem: [V+1][R*Wf] floats + u16 table[R*Wv]
template <int V, int NT>
__device__ __forceinline__ void
cv_fwd_unit(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ cost,
            int C, int Df, int Hf, int Wf, int R, int dchunk, int tile, int dci, int c, int b, float* smem) {
    using VT = typename Vec<V>::T;
    const int Wv = Wf / V;
    const int h0 = tile * R;
    const int rows = min(R, Hf - h0);
    const int d0 = dci * dchunk;                 // multiple of V by construction
    const int nd = min(dchunk, Df - d0);
    const int P = rows * Wv;                     // vectors in the tile
    const int tile_elems = R * Wf;

    float* sx = smem;                            // left rows
    float* sy = smem + tile_elems;               // V shifted copies of the right rows
    unsigned short* wvtab = reinterpret_cast<unsigned short*>(smem + (V + 1) * tile_elems);

    // ---- stage the rows (each input element read once per CTA) ----
    const size_t in_off = ((size_t)(b * C + c) * Hf + h0) * Wf;
    const VT* xg = reinterpret_cast<const VT*>(x + in_off);
    const VT* yg = reinterpret_cast<const VT*>(y + in_off);
    for (int p = threadIdx.x; p < P; p += NT) {
        const int r = p / Wv;
        const int wv = p - r * Wv;
        wvtab[p] = (unsigned short)wv;
        reinterpret_cast<VT*>(sx)[p] = __ldg(xg + p);
        const VT yv = __ldg(yg + p);
        const int w0 = wv * V;
#pragma unroll
        for (int s = 0; s < V; ++s) {
            float* row = sy + s * tile_elems + r * Wf;
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const int i = w0 + k + s;        // copy_s[i] = y[i - s]
                if (i < Wf) row[i] = get(yv, k);
            }
            if (wv == 0) {
#pragma unroll
                for (int k = 0; k < V; ++k)
                    if (k < s) row[k] = 0.f;     // copy_s[i < s] = 0
            }
        }
    }
    __syncthreads();

    // ---- stream the volume: items = (d_local, p), consecutive threads -> consecutive vectors ----
    const size_t plane = (size_t)Hf * Wf;
    float* left = cost + (((size_t)(b * 2 * C + c) * Df + d0) * Hf + h0) * Wf;
    float* right = left + (size_t)C * Df * plane;
    const VT* sxv = reinterpret_cast<const VT*>(sx);

    int p = threadIdx.x, dl = 0;
    while (p >= P) { p -= P; ++dl; }
    while (dl < nd) {
        const int d = d0 + dl;
        const int wv = wvtab[p];
        const int w0 = wv * V;
        const size_t off = (size_t)dl * plane + (size_t)p * V;
        // left half: x masked by w >= d
        VT xv = sxv[p];
        if (w0 < d) {
#pragma unroll
            for (int k = 0; k < V; ++k)
                if (w0 + k < d) set(xv, k, 0.f);
        }
        st_stream(reinterpret_cast<VT*>(left + off), xv);
        // right half: y shifted by d = V*q + s  ->  copy s, vector (wv - q)
        const int q = d / V, s = d - q * V;
        VT yv = zero_vec<VT>();
        if (wv >= q) yv = reinterpret_cast<const VT*>(sy + s * tile_elems)[p - q];
        st_stream(reinterpret_cast<VT*>(right + off), yv);
        p += NT;
        while (p >= P) { p -= P; ++dl; }
    }
}

// grid: x = h-tile * n_dchunks + d-chunk, y = c, z = b.
template <int V, int NT>
__global__ void __launch_bounds__(NT)
cv_fwd_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ cost,
              int C, int Df, int Hf, int Wf, int R, int dchunk, int n_dchunks) {
    extern __shared__ __align__(16) float smem[];
    const int tile = blockIdx.x / n_dchunks;
    cv_fwd_unit<V, NT>(x, y, cost, C, Df, Hf, Wf, R, dchunk, tile, blockIdx.x - tile * n_dchunks, blockIdx.y, blockIdx.z, smem);
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// Vector path (Wf % 4 == 0): one thread owns vector p of the (b, c) plane.
template <int U>
__device__ __forceinline__ void cv_bwd_v4_unit(const float* __restrict__ g, float* __restrict__ gx, float* __restrict__ gy,
                                               int C, int Df, int Wv, int PV, int p, int c, int b) {
    const int wv = p % Wv;
    const int w0 = wv << 2;
    const size_t planeV = (size_t)PV;
    const float4* gl = reinterpret_cast<const float4*>(g) + (size_t)(b * 2 * C + c) * Df * planeV + p;
    const float4* gr = gl + (size_t)C * Df * planeV;

    float4 ax = make_float4(0.f, 0.f, 0.f, 0.f), ay = ax;
    // d runs from the first multiple-of-4 boundary above Df-1 down to 0 in blocks of U (4 or 2) so that
    // s = d & 3 is a compile-time constant inside the unrolled body
    for (int dq = ((Df + 3) & ~3) - 1; dq >= 0; dq -= U) {
        float4 tl[U], ta[U], tb[U];
        const int q = dq >> 2;                      // same q for the U disparities of this block
        const bool inA = (wv + q) < Wv;
        const bool inB = (wv + q + 1) < Wv;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int d = dq - u;
            const bool dv = d < Df;
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            tl[u] = (dv && (w0 + 3 >= d)) ? ld_stream(gl + (size_t)d * planeV) : z;
            ta[u] = (dv && inA) ? __ldg(gr + (size_t)d * planeV + q) : z;
            tb[u] = (dv && inB && ((U == 4 ? 3 - u : (d & 3)) > 0)) ? __ldg(gr + (size_t)d * planeV + q + 1) : z;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int d = dq - u;
            if (d < Df) {
                // gx[w] += g[d][w] for w >= d
                if (w0 + 0 >= d) ax.x = ax.x + tl[u].x;
                if (w0 + 1 >= d) ax.y = ax.y + tl[u].y;
                if (w0 + 2 >= d) ax.z = ax.z + tl[u].z;
                if (w0 + 3 >= d) ax.w = ax.w + tl[u].w;
                // gy[w'] += g[d][w'+d], elements s..s+3 of the 8-float window (A,B), s = 3-u
                if (inA) {
                    const int s = (U == 4) ? 3 - u : (d & 3);
                    const float e0 = s == 0 ? ta[u].x : s == 1 ? ta[u].y : s == 2 ? ta[u].z : ta[u].w;
                    const float e1 = s == 0 ? ta[u].y : s == 1 ? ta[u].z : s == 2 ? ta[u].w : tb[u].x;
                    const float e2 = s == 0 ? ta[u].z : s == 1 ? ta[u].w : s == 2 ? tb[u].x : tb[u].y;
                    const float e3 = s == 0 ? ta[u].w : s == 1 ? tb[u].x : s == 2 ? tb[u].y : tb[u].z;
                    // validity: w'+d < Wf  <=>  element index (s+k) stays inside A, or B exists
                    ay.x = ay.x + e0;                                   // s+0 <= 3: always inside A
                    if (s + 1 <= 3 || inB) ay.y = ay.y + e1;
                    if (s + 2 <= 3 || inB) ay.z = ay.z + e2;
                    if (s + 3 <= 3 || inB) ay.w = ay.w + e3;
                }
            }
        }
    }
    const size_t o = (size_t)(b * C + c) * planeV + p;
    reinterpret_cast<float4*>(gx)[o] = ax;
    reinterpret_cast<float4*>(gy)[o] = ay;
}

// grid: x over Hf*Wv vectors, y = c, z = b.
template <int NT, int U, int MINB>
__global__ void __launch_bounds__(NT, MINB)
cv_bwd_v4_kernel(const float* __restrict__ g, float* __restrict__ gx, float* __restrict__ gy,
                 int C, int Df, int Hf, int Wf) {
    const int Wv = Wf >> 2;
    const int PV = Hf * Wv;
    const int p = blockIdx.x * NT + threadIdx.x;
    if (p >= PV) return;
    cv_bwd_v4_unit<U>(g, gx, gy, C, Df, Wv, PV, p, blockIdx.y, blockIdx.z);
}

// Persistent form: a grid of `per_sm` CTAs per SM that is resident at once walks the items (b*C + c, block of NT vectors)
// in order.  Used when the kernel has to SHARE the SMs with the FP32-bound head backward on a second stream
// (rag_b200.pipeline.OverlappedTrainPath): launched first, its small footprint (NT threads x ~48 registers per CTA)
// leaves the register file to the head's CTAs, which the block scheduler can then dispatch beside it.
template <int NT, int U>
__global__ void __launch_bounds__(NT)
cv_bwd_v4_persistent_kernel(const float* __restrict__ g, float* __restrict__ gx, float* __restrict__ gy,
                            int BC, int C, int Df, int Hf, int Wf, int n_blk) {
    const int Wv = Wf >> 2;
    const int PV = Hf * Wv;
    const long long n_items = (long long)BC * n_blk;
    for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int bc = (int)(item / n_blk), blk = (int)(item - (long long)bc * n_blk);
        const int p = blk * NT + threadIdx.x;
        if (p < PV) cv_bwd_v4_unit<U>(g, gx, gy, C, Df, Wv, PV, p, bc % C, bc / C);
    }
}

// RAG_CV_BWD_SLIM: the same sums with the in-flight bytes in SHARED MEMORY instead of registers.  The vector kernel
// above keeps 12 x 16 bytes per thread in flight in 48 registers, so saturating HBM takes ~37 K registers per SM and
// the FP32-bound head backward (128 registers x 128 threads per CTA) finds room for one CTA beside it.  Here a CTA of NT
// threads streams its items (b*C + c, block of NT vectors) through a ring of S stages of four disparities each with
// cp.async (LDGSTS: global -> shared, no register staging): ~(S-1) x 4 x (2 NT + 1) x 16 bytes in flight per CTA at
// 64 registers per thread, i.e. ONE 256-thread CTA per SM (a quarter of the register file, 96 KB in flight) carries the
// read stream and three head-backward CTAs fit beside it.  The ring runs across item boundaries (stage n of the CTA's flattened (item, q) sequence), one block barrier
// per stage.  Same arithmetic as cv_bwd_v4_unit -- per output element a sequential fp32 sum over d descending, the same
// predicates -- so the result is bit-identical.
// shared: float4 [S][4][2 NT + 2]: per disparity NT left vectors | NT + 1 right vectors (the block's window shifted by q) | pad
template <int NT, int S>
__global__ void __launch_bounds__(NT)
cv_bwd_staged_kernel(const float* __restrict__ g, float* __restrict__ gx, float* __restrict__ gy,
                     int BC, int C, int Df, int Hf, int Wf, int n_blk) {
    constexpr int ROW = 2 * NT + 2;
    extern __shared__ __align__(16) float4 cbs_smem[];
    const int t = threadIdx.x;
    const int Wv = Wf >> 2, PV = Hf * Wv, nq = (Df + 3) >> 2;
    const long long n_items = (long long)BC * n_blk;
    if ((long long)blockIdx.x >= n_items) return;
    const int n_my = (int)((n_items - blockIdx.x + gridDim.x - 1) / gridDim.x);
    const float4* gv = reinterpret_cast<const float4*>(g);
    const size_t PV4 = (size_t)4 * PV;

    // ---- producer side: the CTA's stages in order -- items blockIdx.x + k * gridDim.x, inside an item q = nq-1 .. 0
    // (disparities 4q .. 4q+3).  All per-stage state advances incrementally: no division outside the item set-up.
    int i_left = n_my * nq, i_slot = 0, i_q = 0, i_wv = 0, i_wvx = 0, i_p = 0, i_px = 0;
    long long i_item = (long long)blockIdx.x - gridDim.x;
    const float4* i_pl = gv;      // left  vector p       of disparity 4 i_q
    const float4* i_pr = gv;      // right vector p + i_q of disparity 4 i_q
    const float4* i_prx = gv;     // right vector (block end) + i_q: the window's extra vector, fetched by thread 0
    auto issue_item = [&]() {
        i_item += gridDim.x;
        const int bc = (int)(i_item / n_blk), blk = (int)(i_item - (long long)bc * n_blk);
        const int b = bc / C, c = bc - b * C;
        i_p = blk * NT + t;
        i_wv = i_p % Wv;
        i_px = blk * NT + NT;
        i_wvx = i_px % Wv;
        i_q = nq - 1;
        const float4* gl = gv + (size_t)(b * 2 * C + c) * Df * PV + (size_t)i_q * PV4;
        i_pl = gl + i_p;
        i_pr = gl + (size_t)C * Df * PV + i_p + i_q;
        i_prx = gl + (size_t)C * Df * PV + i_px + i_q;
    };
    issue_item();
    auto issue = [&]() {
        if (i_left > 0) {
            float4* st = cbs_smem + (size_t)i_slot * 4 * ROW;
            const bool lf = i_p < PV && i_q <= i_wv;                     // some w of the vector has w >= d in this stage
            const bool rA = i_p + i_q < PV && i_wv + i_q < Wv;          // vector p + q is somebody's in-row "A" or "B" vector
            const bool rX = t == 0 && i_px + i_q < PV && i_wvx + i_q < Wv;
            const int nd = min(4, Df - 4 * i_q);
#pragma unroll
            for (int dd = 0; dd < 4; ++dd) {
                if (dd < nd) {
                    if (lf) __pipeline_memcpy_async(st + dd * ROW + t, i_pl + (size_t)dd * PV, 16);
                    if (rA) __pipeline_memcpy_async(st + dd * ROW + NT + t, i_pr + (size_t)dd * PV, 16);
                    if (rX) __pipeline_memcpy_async(st + dd * ROW + 2 * NT, i_prx + (size_t)dd * PV, 16);
                }
            }
            --i_left;
            i_slot = i_slot + 1 == S ? 0 : i_slot + 1;
            if (i_q == 0) {
                if (i_left > 0) issue_item();
            } else {
                --i_q;
                i_pl -= PV4; i_pr -= PV4 + 1; i_prx -= PV4 + 1;
            }
        }
        __pipeline_commit();
    };
#pragma unroll 1
    for (int n = 0; n < S - 1; ++n) issue();

    // ---- consumer side ----
    float4 ax = make_float4(0.f, 0.f, 0.f, 0.f), ay = ax;
    int c_wv = 0, c_q = 0, c_slot = 0;
    bool c_valid = false;
    size_t c_out = 0;
    long long c_item = (long long)blockIdx.x - gridDim.x;
#pragma unroll 1
    for (int n = n_my * nq; n > 0; --n) {
        if (c_q == 0) {                                   // first stage of the next item
            c_item += gridDim.x;
            const int bc = (int)(c_item / n_blk), blk = (int)(c_item - (long long)bc * n_blk);
            const int p = blk * NT + t;
            c_valid = p < PV;
            c_wv = p % Wv;
            c_out = (size_t)bc * PV + p;
            c_q = nq;
            ax = make_float4(0.f, 0.f, 0.f, 0.f);
            ay = ax;
        }
        --c_q;
        __pipeline_wait_prior(S - 2);                 // this thread's copies of the stage have landed ...
        __syncthreads();                              // ... and everybody's; the previous stage is consumed
        issue();                                      // refills the previous stage's buffer
        const float4* st = cbs_smem + (size_t)c_slot * 4 * ROW;
        c_slot = c_slot + 1 == S ? 0 : c_slot + 1;
        const bool inA = c_valid && (c_wv + c_q) < Wv;
        const bool inB = c_valid && (c_wv + c_q + 1) < Wv;
        const bool lf = c_valid && c_q <= c_wv;
        const bool diag = c_q == c_wv;                // the vector straddles w == d: element e counts when e >= d & 3
        const int nd = min(4, Df - 4 * c_q);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int sft = 3 - u;                    // d = 4 c_q + sft, descending
            if (sft < nd) {
                if (lf) {
                    const float4 tl = st[sft * ROW + t];
                    if (!diag || sft <= 0) ax.x = ax.x + tl.x;
                    if (!diag || sft <= 1) ax.y = ax.y + tl.y;
                    if (!diag || sft <= 2) ax.z = ax.z + tl.z;
                    ax.w = ax.w + tl.w;
                }
                if (inA) {
                    const float4 ta = st[sft * ROW + NT + t];
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 tb = (inB && sft > 0) ? st[sft * ROW + NT + t + 1] : z;
                    const float e0 = sft == 0 ? ta.x : sft == 1 ? ta.y : sft == 2 ? ta.z : ta.w;
                    const float e1 = sft == 0 ? ta.y : sft == 1 ? ta.z : sft == 2 ? ta.w : tb.x;
                    const float e2 = sft == 0 ? ta.z : sft == 1 ? ta.w : sft == 2 ? tb.x : tb.y;
                    const float e3 = sft == 0 ? ta.w : sft == 1 ? tb.x : sft == 2 ? tb.y : tb.z;
                    ay.x = ay.x + e0;
                    if (sft + 1 <= 3 || inB) ay.y = ay.y + e1;
                    if (sft + 2 <= 3 || inB) ay.z = ay.z + e2;
                    if (sft + 3 <= 3 || inB) ay.w = ay.w + e3;
                }
            }
        }
        if (c_q == 0 && c_valid) {
            reinterpret_cast<float4*>(gx)[c_out] = ax;
            reinterpret_cast<float4*>(gy)[c_out] = ay;
        }
    }
}

// Scalar path (any Wf).  grid: x over Hf*Wf elements, y = c, z = b.
template <int NT>
__global__ void __launch_bounds__(NT)
cv_bwd_scalar_kernel(const float* __restrict__ g, float* __restrict__ gx, float* __restrict__ gy,
                     int C, int Df, int Hf, int Wf) {
    const int PE = Hf * Wf;
    const int p = blockIdx.x * NT + threadIdx.x;
    if (p >= PE) return;
    const int c = blockIdx.y, b = blockIdx.z;
    const int w = p % Wf;
    const float* gl = g + (size_t)(b * 2 * C + c) * Df * PE + p;
    const float* gr = gl + (size_t)C * Df * PE;
    float ax = 0.f, ay = 0.f;
    for (int d = Df - 1; d >= 0; --d) {
        if (w >= d) ax = ax + ld_stream(gl + (size_t)d * PE);
        if (w + d < Wf) ay = ay + ld_stream(gr + (size_t)d * PE + d);
    }
    const size_t o = (size_t)(b * C + c) * PE + p;
    gx[o] = ax;
    gy[o] = ay;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static int check_cv_args(const void* a, const void* b_, const void* c, int B, int C, int Df, int Hf, int Wf) {
    if (!a || !b_ || !c) return fail(RAG_E_NULL, "cost_volume: null pointer");
    if (B <= 0 || C <= 0 || Df <= 0 || Hf <= 0 || Wf <= 0)
        return fail(RAG_E_SHAPE, "cost_volume: non-positive dimension B=%d C=%d Df=%d Hf=%d Wf=%d", B, C, Df, Hf, Wf);
    if (B > 65535 || C > 65535) return fail(RAG_E_SHAPE, "cost_volume: B and C must be <= 65535");
    // the kernels index (b*2C + c) and the item count B*C*tiles*chunks in 32-bit int
    if ((long long)2 * B * C >= (1LL << 31) || (long long)B * C * Hf * ((Df + 15) / 16) >= (1LL << 31))
        return fail(RAG_E_SHAPE, "cost_volume: 2*B*C and B*C*Hf*ceil(Df/16) must be < 2^31");
    if ((size_t)Df * Hf * Wf >= ((size_t)1 << 31) || Wf > 65535)
        return fail(RAG_E_SHAPE, "cost_volume: Df*Hf*Wf must be < 2^31 and Wf <= 65535");
    if (!aligned(a, 4) || !aligned(b_, 4) || !aligned(c, 4)) return fail(RAG_E_ALIGN, "cost_volume: pointers must be 4-byte aligned");
    return RAG_OK;
}

// any width / alignment: items (d, vector) dealt to threads, 16-disparity chunks, 36 KB tiles
template <int V, int NT>
static int launch_cv_fwd(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf, cudaStream_t st) {
    int dchunk = ((16 + V - 1) / V) * V;
    const int n_dchunks = (Df + dchunk - 1) / dchunk;
    const size_t budget = 36 * 1024;
    int R = (int)(budget / ((size_t)(V + 1) * 4 * Wf + (size_t)2 * (Wf / V)));
    R = R < 1 ? 1 : (R > Hf ? Hf : R);
    // prefer an R that divides Hf (no ragged last tile) when one is close
    for (int r = R; r >= (R * 3) / 4 && r >= 1; --r)
        if (Hf % r == 0) { R = r; break; }
    const size_t smem = (size_t)(V + 1) * R * Wf * 4 + (size_t)R * (Wf / V) * 2;
    if (smem > 200 * 1024) return fail(RAG_E_SHAPE, "cost_volume_fwd: Wf=%d too wide for one shared-memory row tile", Wf);
    auto kern = cv_fwd_kernel<V, NT>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail((int)e, "cost_volume_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    const int n_tiles = (Hf + R - 1) / R;
    if ((long long)n_tiles * n_dchunks > 2147483647LL) return fail(RAG_E_SHAPE, "cost_volume_fwd: grid too large");
    dim3 grid(n_tiles * n_dchunks, C, B);
    kern<<<grid, NT, smem, st>>>(x, y, cost, C, Df, Hf, Wf, R, dchunk, n_dchunks);
    return check_launch("cost_volume_fwd");
}

static bool cv_lean_ok(const float* x, const float* y, const float* cost, int Wf) {
    return Wf % 4 == 0 && Wf <= 2048 && aligned(x, 16) && aligned(y, 16) && aligned(cost, 16);
}

// zero the caller's work counter on the launch stream (stream-ordered before the kernel that consumes it)
static int arm_counter(void* workspace, cudaStream_t st, const char* who) {
    if (!aligned(workspace, 8)) return fail(RAG_E_ALIGN, "%s: workspace must be 8-byte aligned", who);
    cudaError_t e = cudaMemsetAsync(workspace, 0, RAG_CV_FWD_WORKSPACE_BYTES, st);
    if (e != cudaSuccess) return fail((int)e, "%s: cudaMemsetAsync(workspace): %s", who, cudaGetErrorString(e));
    return RAG_OK;
}

// lean thread-stationary kernel.  !DYN: one CTA per item (hardware dispatch order keeps the resident CTAs on
// neighbouring rows; stateless; ctr unused).  DYN: persistent grid of `per_sm` CTAs per SM that takes its items IN
// ORDER from the caller's counter `ctr` (3 % faster at B=8 480x960, and resident at once, which is what lets the
// disparity head share the SMs on a second stream).
template <int NT, int VPT, bool DYN>
static int launch_cv_fwd_lean(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf,
                              int per_sm, unsigned int* ctr, cudaStream_t st, int dchunk_max = 16) {
    const int Wv = Wf / 4, Df4 = (Df + 3) & ~3;
    const size_t row_bytes = (size_t)16 * (Df4 + Wf + 4);          // four images of one row
    int R = std::min(Hf, (NT * VPT) / Wv);
    if (R < 1) return fail(RAG_E_SHAPE, "cost_volume_fwd(lean): Wf=%d too wide for a %d-vector tile", Wf, NT * VPT);
    while (R > 1 && R * row_bytes > 64 * 1024) --R;
    const size_t smem = R * row_bytes;
    if (smem > 200 * 1024) return fail(RAG_E_SHAPE, "cost_volume_fwd(lean): Df=%d Wf=%d do not fit shared memory", Df, Wf);
    auto kern = cv_fwd_lean_kernel<NT, VPT, DYN>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    // the L1/shared split of an SM cannot change while CTAs are resident: ask for the largest shared-memory
    // carve-out so that this kernel and the disparity head (which does the same) can share an SM
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return fail((int)e, "cost_volume_fwd(lean): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int n_tiles = (Hf + R - 1) / R;
    const int dchunk = std::min(dchunk_max, (Df + 3) & ~3);
    const int n_dchunks = (Df + dchunk - 1) / dchunk;
    const long long n_items = (long long)B * C * n_tiles * n_dchunks;
    if (n_items >= (1LL << 31)) return fail(RAG_E_SHAPE, "cost_volume_fwd(lean): too many work items");
    const int grid = (int)(DYN ? std::min<long long>(n_items, (long long)num_sms() * per_sm) : n_items);
    if (DYN) if (int rc = arm_counter(ctr, st, "cost_volume_fwd(lean)")) return rc;
    kern<<<grid, NT, smem, st>>>(x, y, cost, B * C, C, Df, Hf, Wf, R, n_tiles, dchunk, n_dchunks, ctr);
    return check_launch("cost_volume_fwd(lean)");
}

// variant: -1 = default (lean persistent (variant 5) when a workspace is given, lean one-CTA-per-item without, generic when the
// lean preconditions fail); 0 = generic; 1 = lean one CTA per item; 3 = lean persistent 512 threads, RAG_CV_FWD_SHARED (needs
// workspace); 5 = lean persistent 256 threads x 1 vector, RAG_CV_FWD_SLIM (needs workspace).  Ids 2 (lean persistent 256
// threads x 2 vectors) and 4 (TMA bulk stores) were retired: slower than 5 on every measured shape (DESIGN.md section 5.1).
int cost_volume_fwd(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf,
                    void* workspace, int variant, cudaStream_t st) {
    if (int e = check_cv_args(x, y, cost, B, C, Df, Hf, Wf)) return e;
    if (variant < -1 || variant > 5 || variant == 2 || variant == 4)
        return fail(RAG_E_VARIANT, "cost_volume_fwd: unknown variant %d (ids 2 and 4 were retired)", variant);
    unsigned int* ctr = static_cast<unsigned int*>(workspace);
    const bool lean = cv_lean_ok(x, y, cost, Wf) && (Wf / 4) <= 512;
    if (variant == -1) variant = lean ? (ctr ? RAG_CV_FWD_SLIM : 1) : 0;   // the slim geometry is also the fastest alone
    if (variant >= 3 && !ctr) return fail(RAG_E_NULL, "cost_volume_fwd: variant %d needs a workspace of RAG_CV_FWD_WORKSPACE_BYTES", variant);
    if (variant >= 1 && !lean)
        return fail(RAG_E_VARIANT, "cost_volume_fwd: lean variants need Wf %% 4 == 0, Wf <= 2048 and 16-byte aligned pointers");
    if (variant == 1) return launch_cv_fwd_lean<256, 2, false>(x, y, cost, B, C, Df, Hf, Wf, 0, nullptr, st);
    if (variant == 3) return launch_cv_fwd_lean<512, 1, true>(x, y, cost, B, C, Df, Hf, Wf, 1, ctr, st);
    // RAG_CV_FWD_SLIM: 256 threads x 1 vector (at most 64 registers: a quarter of the register file per SM), 32 disparities per item
    if (variant == 5) return launch_cv_fwd_lean<256, 1, true>(x, y, cost, B, C, Df, Hf, Wf, 1, ctr, st, 32);
    const bool a16 = aligned(x, 16) && aligned(y, 16) && aligned(cost, 16);
    const bool a8 = aligned(x, 8) && aligned(y, 8) && aligned(cost, 8);
    if (Wf % 4 == 0 && a16) return launch_cv_fwd<4, 256>(x, y, cost, B, C, Df, Hf, Wf, st);
    if (Wf % 2 == 0 && a8) return launch_cv_fwd<2, 256>(x, y, cost, B, C, Df, Hf, Wf, st);
    return launch_cv_fwd<1, 256>(x, y, cost, B, C, Df, Hf, Wf, st);
}

// variant: 0 = default (128-bit vector kernel when Wf % 4 == 0 and aligned, else scalar); 1 = scalar;
// 2 = RAG_CV_BWD_SHARED: the vector kernel as a persistent grid of 4 x 128-thread CTAs per SM (SM sharing);
// 3 = RAG_CV_BWD_SLIM: cp.async ring in shared memory, one 256-thread CTA per SM with 4 stages (3 stages: 0.078 instead of
// 0.076 ms at B=4 288x576; 128 threads x 6 stages: 0.119 ms -- profiles/r2_coresident_sweep_288x576_b4.jsonl)
int cost_volume_bwd(const float* g, float* gx, float* gy, int B, int C, int Df, int Hf, int Wf,
                    int variant, cudaStream_t st) {
    if (int e = check_cv_args(g, gx, gy, B, C, Df, Hf, Wf)) return e;
    if (variant < 0 || variant > 3) return fail(RAG_E_VARIANT, "cost_volume_bwd: unknown variant %d", variant);
    const bool a16 = aligned(g, 16) && aligned(gx, 16) && aligned(gy, 16);
    if (variant >= 2) {
        if (!(Wf % 4 == 0 && a16)) return fail(RAG_E_VARIANT, "cost_volume_bwd: variant %d needs Wf %% 4 == 0 and 16-byte aligned pointers", variant);
        constexpr int NT = 128;
        const int PV = Hf * (Wf / 4), n_blk = (PV + NT - 1) / NT;
        const long long n_items = (long long)B * C * n_blk;
        if (variant == 3) {   // RAG_CV_BWD_SLIM: cp.async ring in shared memory, one CTA per SM
            auto launch = [&](auto kern, int nt, int stages) -> int {
                const size_t smem = (size_t)stages * 4 * (2 * nt + 2) * sizeof(float4);
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
                if (e != cudaSuccess) return fail((int)e, "cost_volume_bwd(staged): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
                const int nb = (PV + nt - 1) / nt;
                const long long items = (long long)B * C * nb;
                const int grid = (int)std::min<long long>(items, (long long)num_sms());
                kern<<<grid, nt, smem, st>>>(g, gx, gy, B * C, C, Df, Hf, Wf, nb);
                return RAG_OK;
            };
            if (int rc = launch(cv_bwd_staged_kernel<256, 4>, 256, 4)) return rc;
            return check_launch("cost_volume_bwd(staged)");
        }
        const int grid = (int)std::min<long long>(n_items, (long long)num_sms() * 4);
        cv_bwd_v4_persistent_kernel<NT, 4><<<grid, NT, 0, st>>>(g, gx, gy, B * C, C, Df, Hf, Wf, n_blk);
    } else if (variant != 1 && Wf % 4 == 0 && a16) {
        constexpr int NT = 128;
        const int PV = Hf * (Wf / 4);
        dim3 grid((PV + NT - 1) / NT, C, B);
        cv_bwd_v4_kernel<NT, 4, 1><<<grid, NT, 0, st>>>(g, gx, gy, C, Df, Hf, Wf);
    } else {
        constexpr int NT = 256;
        const int PE = Hf * Wf;
        dim3 grid((PE + NT - 1) / NT, C, B);
        cv_bwd_scalar_kernel<NT><<<grid, NT, 0, st>>>(g, gx, gy, C, Df, Hf, Wf);
    }
    return check_launch("cost_volume_bwd");
}

}  // namespace rag
