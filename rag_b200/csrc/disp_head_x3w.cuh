// x3 disparity-head backward, second generation (the default whenever maxdisp == 3*Dl: <RED = true>).
//
// Same maths as head_bwd_x3_kernel (disp_head_x3.cuh): deterministic, atomics-free transpose of the
// upsample applied to -g p_k (k - disp), p_k rebuilt from cost_lr and the forward's stats.  What the
// profile of the first kernel showed (profiles/r1_train_bwd_kernels_ncu.md): 111 M warp instructions
// for a batch the forward does in 26 M -- issue bound at 69 %, 1.5 waves of long tasks, 25 % of the work
// recomputed halo rows.  So here
//   * a task is ONE block row (no halo rows): its "A" part (cell row rb) goes to gcost, its "B" part
//     (cell row rb+1) to a scratch buffer of the same shape, and a trivial second kernel adds the two in a
//     fixed order (still deterministic) -- 5x more, 5x shorter tasks and no recomputation;
//   * the warp's 2 x 34 x (J+2) low-res window is staged in shared memory with cp.async, so the k-block
//     loop reads it at compile-time offsets;
//   * the per-bin arithmetic runs on packed FP32 (FFMA2/FMUL2) with the pixel pairing of the forward
//     (P0=(p00,p01) P1=(p10,p11) P2=(p20,p21) P3=(p02,p12) S=p22).
// CTA-tasks: ceil(Wl/31) strips x ceil((Hl+1)*nJ / 4) task groups x B; 128 threads (4 independent warp tasks).
#pragma once
#include <cuda_pipeline.h>

#include "disp_head_x3.cuh"

namespace rag {

constexpr int kBwJ = 16;                 // low-res bins (cells) per task
constexpr int kBwBins = kBwJ + 2;        // low-res bins a task reads
constexpr int kBwCols = 34;              // window width: 32 block columns + 1 + pad
constexpr int kBwWin = kBwBins * 2 * kBwCols;

//
// Cube root: the three full-res bins of a k-block come from ONE exp2 per pixel instead of three.  With
// c_j = 2^(e_j/3) (e_j = relative exponent of low-res bin j) and PyTorch's lambdas (0, ~1/3, ~2/3),
//   2^e(3j+1) = c_j^3,   2^e(3j+2) = c_j^2 c_j+1 (1 + kap2 du),   2^e(3j+3) = c_j c_j+1^2 (1 + kap3 du),
// du = (e_j+1 - e_j)/3, kap_q = 3 ln2 (lambda_fp32 - q/3): the first-order term restores the reference's
// fp32 lambdas (|kap du| < 2e-4 wherever the bin matters, so the second order is < 2e-8).  The profile of
// the three-exp2 form had the XU pipe 45 % and the FMA pipe 56 % busy with the issue slots at 63 %: the
// MUFU bursts (27 per k-block, 8 clk each) were what the four warps of a scheduler queued on.
//
// RED: both parts are added straight into a ZEROED gcost with red.global.add.f32 -- no scratch buffer, no
// combine kernel.  Every element receives exactly two contributions (its row's "A" part and the row
// above's "B" part); 0 + a + b and 0 + b + a are the same fp32 value (addition is commutative and 0 + a is
// exact), so the result does not depend on the order the two arrive in: still bitwise deterministic.
// (red.global.add.f32 flushes subnormal addends and sums to zero, as PyTorch's own atomicAdd backward does;
// against the scratch + combine variant the result differs at most by that and by the sign of a zero.)
//
// Grid.  Default: 3-D, one CTA per CTA-task (strip, group of 4 warp tasks, image).  <PERSIST>: 1-D, CTA blockIdx.x walks the
// flattened CTA-tasks ct = (b * ny + group) * strips + strip, ny = ceil(n_tasks / 4), with stride gridDim.x -- a grid of a
// few CTAs per SM that is resident at once, which is what lets the kernel share the SMs with a cost-volume kernel on
// another stream whichever of the two is launched first (RAG_HEAD_BWD_SHARED, rag_b200.pipeline).  The warps of a CTA
// walk their task lists independently: the depth tables are built once per CTA, nothing else is shared between tasks.
template <bool RED, bool PERSIST = false>
__global__ void __launch_bounds__(128, 4)
head_bwd_x3w_kernel(const float* __restrict__ cost, const float* __restrict__ gdisp, const float* __restrict__ disp,
                    const float* __restrict__ stats, float* __restrict__ gcost, float* __restrict__ scratch,
                    int Dl, int Hl, int Wl, float scale, int nJ, int n_tasks, int strips, int n_ct) {
    extern __shared__ __align__(16) float x3w_smem[];
    const int D = 3 * Dl, H = 3 * Hl, W = 3 * Wl;
    float2* lzb = reinterpret_cast<float2*>(x3w_smem);   // [D+3] kap_q of bin k (see above), broadcast
    float2* dAb = lzb + (D + 3);                          // [D+3] weight of bin k into cell (k-1)/3, broadcast
    float2* dBb = dAb + (D + 3);                          // [D+3] ... into cell (k-1)/3 + 1
    float* win_all = reinterpret_cast<float*>(dBb + (D + 3));
    for (int k = threadIdx.x; k < D + 3; k += 128) {
        float l0 = 0.f, l1 = 0.f, wa = 0.f, wb = 0.f;
        if (k < D) {
            int t0, t1;
            src_index<true>(scale, k, Dl, t0, t1, l0, l1);
            const int jb = k == 0 ? 0 : (k - 1) / 3;
            wa = (t0 == jb ? l0 : 0.f) + (t1 == jb ? l1 : 0.f);
            wb = (t0 == jb + 1 ? l0 : 0.f) + (t1 == jb + 1 ? l1 : 0.f);
            // lambda - fl(q/3) is exact in fp32 (Sterbenz); fl(1/3) - 1/3 = 2^-25/3, fl(2/3) - 2/3 = 2^-24/3
            const int q = k == 0 ? 0 : (k - 1) % 3;
            const float third = q == 1 ? 0.333333343267440796f : 0.666666686534881592f;
            const float resid = q == 1 ? 9.934107e-9f : 1.9868214e-8f;
            l1 = (q != 0 && t1 > t0) ? 2.0794415416798357f * ((l1 - third) + resid) : 0.f;
        }
        lzb[k] = f2b(l1); dAb[k] = f2b(wa); dBb[k] = f2b(wb);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* win = win_all + warp * kBwWin;
    const int ny = (n_tasks + 3) >> 2;
    int ct = blockIdx.x;
    do {                                                  // !PERSIST: exactly one pass, the loop folds away
    // !PERSIST: 3-D grid (strip, task group, image); PERSIST: 1-D grid over the flattened CTA-tasks
    const int cq = PERSIST ? ct / strips : 0;
    const int strip = PERSIST ? ct - cq * strips : (int)blockIdx.x;
    const int b = PERSIST ? cq / ny : (int)blockIdx.z;
    const int task = (PERSIST ? cq - b * ny : (int)blockIdx.y) * 4 + warp;
    if (task >= n_tasks) continue;
    __syncwarp();                                         // the previous task's window reads are done
    const int rbi = task / nJ, jc = task - rbi * nJ;
    const int rb = rbi - 1;                               // block row, -1 .. Hl-1
    const int j0 = jc * kBwJ, j1 = min(j0 + kBwJ, Dl);
    const int jb0 = max(j0 - 1, 0);                       // first k-block (its B part feeds cell j0)
    const int c_first = strip * 31 - 1;
    const int c_raw = c_first + lane;
    const bool lane_on = c_raw <= Wl - 1;
    const int c = min(c_raw, Wl - 1);

    X3Axis aw, ah;
    x3_axis(scale, c, Wl, aw);
    if (!lane_on) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { aw.wa[i] = 0.f; aw.wb[i] = 0.f; aw.valid[i] = false; }
    }
    x3_axis(scale, rb, Hl, ah);
    const size_t plane = (size_t)Hl * Wl;
    const size_t img = (size_t)H * W;
    const float* base = cost + (size_t)b * Dl * plane;

    // ---- stage the window: bins jb0..min(j1,Dl-1), rows (lo0, lo1), columns clamp(c_first + u), u = 0..33 ----
    {
        const int nb = min(j1, Dl - 1) - jb0 + 1;
        const int gc0 = min(max(c_first + lane, 0), Wl - 1);
        const int gc32 = min(max(c_first + 32, 0), Wl - 1), gc33 = min(max(c_first + 33, 0), Wl - 1);
        // lanes 0,1 fetch the two extra columns in a second pass, so that every copy is one running pointer
        const float* s0 = base + (size_t)jb0 * plane + (size_t)ah.lo0 * Wl + gc0;
        const float* s1 = base + (size_t)jb0 * plane + (size_t)ah.lo1 * Wl + gc0;
        float* d = win + lane;
#pragma unroll 2
        for (int q = 0; q < nb; ++q) {
            __pipeline_memcpy_async(d, s0, 4);
            __pipeline_memcpy_async(d + kBwCols, s1, 4);
            s0 += plane; s1 += plane; d += 2 * kBwCols;
        }
        if (lane < 4) {
            const float* s2 = base + (size_t)jb0 * plane + (size_t)((lane & 2) ? ah.lo1 : ah.lo0) * Wl + ((lane & 1) ? gc33 : gc32);
            float* d2 = win + ((lane & 2) ? kBwCols : 0) + 32 + (lane & 1);
            for (int q = 0; q < nb; ++q) {
                __pipeline_memcpy_async(d2, s2, 4);
                s2 += plane; d2 += 2 * kBwCols;
            }
        }
        __pipeline_commit();
    }

    // ---- per-pixel data (overlaps the window copy) ----
    const float* gd = gdisp + (size_t)b * img;
    const float* dp = disp + (size_t)b * img;
    const float* sm = stats + (size_t)b * 2 * img;
    float2 mneg[4], gneg[4], dsp[4];
    float mnegS, gnegS, dspS;
    float gabs = 0.f;
    {
        float m9[9], g9[9], d9[9];
#pragma unroll
        for (int ph = 0; ph < 3; ++ph)
#pragma unroll
            for (int pw = 0; pw < 3; ++pw) {
                const int i = ph * 3 + pw;
                const size_t o = (size_t)ah.idx[ph] * W + aw.idx[pw];   // clamped -> always a real pixel
                const bool ok = ah.valid[ph] && aw.valid[pw];
                m9[i] = -__ldg(sm + o) * 0.333333343267440796f;   // the cube-root form works on exponent / 3
                d9[i] = __ldg(dp + o);
                g9[i] = ok ? -__ldg(gd + o) * __ldg(sm + img + o) : 0.f;
                gabs = fmaxf(gabs, fabsf(g9[i]));
            }
#pragma unroll
        for (int ph = 0; ph < 3; ++ph) {
            mneg[ph] = f2(m9[ph * 3], m9[ph * 3 + 1]); gneg[ph] = f2(g9[ph * 3], g9[ph * 3 + 1]); dsp[ph] = f2(d9[ph * 3], d9[ph * 3 + 1]);
        }
        mneg[3] = f2(m9[2], m9[5]); gneg[3] = f2(g9[2], g9[5]); dsp[3] = f2(d9[2], d9[5]);
        mnegS = m9[8]; gnegS = g9[8]; dspS = d9[8];
    }
    float* gout = gcost + (size_t)b * Dl * plane;
    float* sout = (RED ? gcost : scratch) + (size_t)b * Dl * plane;
    const bool store_lane = lane >= 1 && lane_on;
    const bool has_a = rb >= 0;                // cell row rb exists
    const bool has_b = rb + 1 <= Hl - 1;       // cell row rb+1 exists

    // sparse ground truth: no upstream gradient anywhere in the warp's 32 blocks -> zeros, no exp2 work
    if (!__any_sync(0xffffffffu, gabs != 0.f)) {
        __pipeline_wait_prior(0);
        if (store_lane && !RED)
            for (int jb = j0; jb < j1; ++jb) {
                if (has_a) gout[(size_t)jb * plane + (size_t)rb * Wl + c] = 0.f;
                if (has_b) sout[(size_t)jb * plane + (size_t)(rb + 1) * Wl + c] = 0.f;
            }
        continue;
    }

    // packed weights
    const float2 w0p = f2(aw.l0[0], aw.l0[1]), w1p = f2(aw.l1[0], aw.l1[1]);
    const float2 w0c = f2b(aw.l0[2]), w1c = f2b(aw.l1[2]);
    float2 h0b[3], h1b[3], hAb[3], hBb[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        constexpr float ks = kX3NegLog2e / 3.0f;
        h0b[i] = f2b(ah.l0[i] * ks); h1b[i] = f2b(ah.l1[i] * ks);
        hAb[i] = f2b(ah.wa[i]); hBb[i] = f2b(ah.wb[i]);
    }
    const float2 h0p = f2(h0b[0].x, h0b[1].x), h1p = f2(h1b[0].x, h1b[1].x);

    // t = blend(bin at window pointer p) + mneg   (relative exponent of the low-res bin for the 4 pairs + scalar)
    auto blend = [&](const float* p, float2 (&o)[4], float& oS) {
        const float2 v0 = f2b(p[0]), v1 = f2b(p[1]), v2 = f2b(p[kBwCols]), v3 = f2b(p[kBwCols + 1]);
        const float2 x0p = fma2(w0p, v0, mul2(w1p, v1)), x1p = fma2(w0p, v2, mul2(w1p, v3));
        const float2 x0c = fma2(w0c, v0, mul2(w1c, v1)), x1c = fma2(w0c, v2, mul2(w1c, v3));
#pragma unroll
        for (int ph = 0; ph < 3; ++ph) o[ph] = fma2(h0b[ph], x0p, fma2(h1b[ph], x1p, mneg[ph]));
        o[3] = fma2(h0p, x0c, fma2(h1p, x1c, mneg[3]));
        oS = __fmaf_rn(h0b[2].x, x0c.x, __fmaf_rn(h1b[2].x, x1c.x, mnegS));
    };
    // separable transpose of the bilinear blend for one bin part: returns the warp-combined (A row, B row) values
    auto transpose = [&](const float2 (&g)[4], float gS, float& vA, float& vB) {
        const float2 uA = fma2(hAb[2], g[2], fma2(hAb[1], g[1], mul2(hAb[0], g[0])));   // cols 0,1
        const float2 uB = fma2(hBb[2], g[2], fma2(hBb[1], g[1], mul2(hBb[0], g[0])));
        const float uA2 = __fmaf_rn(ah.wa[2], gS, __fmaf_rn(ah.wa[1], g[3].y, ah.wa[0] * g[3].x));   // col 2
        const float uB2 = __fmaf_rn(ah.wb[2], gS, __fmaf_rn(ah.wb[1], g[3].y, ah.wb[0] * g[3].x));
        const float tAA = __fmaf_rn(aw.wa[2], uA2, __fmaf_rn(aw.wa[1], uA.y, aw.wa[0] * uA.x));
        const float tAB = __fmaf_rn(aw.wb[2], uA2, __fmaf_rn(aw.wb[1], uA.y, aw.wb[0] * uA.x));
        const float tBA = __fmaf_rn(aw.wa[2], uB2, __fmaf_rn(aw.wa[1], uB.y, aw.wa[0] * uB.x));
        const float tBB = __fmaf_rn(aw.wb[2], uB2, __fmaf_rn(aw.wb[1], uB.y, aw.wb[0] * uB.x));
        vA = tAA + __shfl_up_sync(0xffffffffu, tAB, 1);    // cell column c: own block's A part + left block's B part
        vB = tBA + __shfl_up_sync(0xffffffffu, tBB, 1);
    };

    __pipeline_wait_prior(0);
    __syncwarp();
    float2 a[4], t[4];
    float aS, tS;
    // running pointers: window slab of the k-block's upper bin, bin tables, output rows
    const float* wp = win + lane;
    const float* wlast = wp + (min(j1, Dl - 1) - jb0) * (2 * kBwCols);
    blend(wp, a, aS);
    const float2* lp = lzb + 3 * jb0 + 1;
    const float2* ap = dAb + 3 * jb0 + 1;
    const float2* bp = dBb + 3 * jb0 + 1;
    float* ga = gout + (size_t)j0 * plane + (size_t)max(rb, 0) * Wl + c;
    float* gb = sout + (size_t)j0 * plane + (size_t)min(rb + 1, Hl - 1) * Wl + c;
    const bool st_a = store_lane && has_a, st_b = store_lane && has_b;
    const float2 neg1 = f2b(-1.f);
    float kf = (float)(3 * jb0 + 1);

    // "B" bin part of the previous k-block, per pixel.  Full-res bin 0 (lambda1 == 0) sits exactly on low-res
    // bin 0 and feeds cell 0 only: its share is the initial value (cell 0 = k-block 0's "A" part + this)
    float2 pg[4] = {f2b(0.f), f2b(0.f), f2b(0.f), f2b(0.f)};
    float pgS = 0.f;
    // c = 2^(a) with a = exponent / 3 of the k-block's lower bin, carried across k-blocks
    float2 ca[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ca[i] = ex2_2(a[i]);
    float caS = ex2_approx(aS);
    if (jb0 == 0 && j0 == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 e0 = mul2(mul2(ca[i], ca[i]), ca[i]);
            pg[i] = mul2(gneg[i], mul2(dAb[0], mul2(e0, fma2(dsp[i], neg1, f2b(0.f)))));
        }
        pgS = gnegS * (dAb[0].x * ((caS * caS * caS) * (0.f - dspS)));
    }
    // the upstream factor -g/sum is folded into (k - disp): gdk = gneg*k - gneg*disp, so the bin terms come out
    // already scaled (two multiplications per pixel pair and k-block fewer)
    float2 ngd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ngd[i] = mul2(mul2(gneg[i], dsp[i]), neg1);
    const float ngdS = -(gnegS * dspS);

#pragma unroll 2
    for (int jb = jb0; jb < j1; ++jb) {
        if (wp < wlast) wp += 2 * kBwCols;   // upper bin min(jb+1, Dl-1)
        blend(wp, t, tS);
        const float2 l2 = lp[1], l3 = lp[2];   // (kap2, kap3); the centre bin lp[0] needs no correction
        const float2 a2 = ap[1], a3 = ap[2];
        const float2 b2 = bp[1], b3 = bp[2];
        lp += 3; ap += 3; bp += 3;
        const float2 kfb = f2b(kf);
        float2 g0[4], g1[4];
        float g0S, g1S;
        // the centre bin k1 = 3 jb + 1 has lambda1 == 0 exactly (it IS low-res bin jb): weight 1 into cell jb,
        // none into cell jb + 1, so its term starts the "A" chain together with the previous k-block's "B" part.
        // Cell jb = this k-block's "A" bin part + the previous k-block's "B" bin part: the spatial transpose is
        // linear, so the two parts are added per pixel first and transposed ONCE
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 ct = ex2_2(t[i]);
            const float2 du = fma2(a[i], neg1, t[i]);
            const float2 x = mul2(ca[i], ct), c2 = mul2(ca[i], ca[i]);
            const float2 dk = fma2(gneg[i], kfb, ngd[i]);        // gneg * (k1 - disp)
            const float2 dk1 = add2(dk, gneg[i]), dk2 = add2(dk1, gneg[i]);
            const float2 q2 = mul2(x, ca[i]), q3 = mul2(x, ct);
            const float2 u2 = mul2(fma2(q2, mul2(l2, du), q2), dk1);
            const float2 u3 = mul2(fma2(q3, mul2(l3, du), q3), dk2);
            g0[i] = fma2(a3, u3, fma2(a2, u2, fma2(mul2(c2, ca[i]), dk, pg[i])));
            g1[i] = fma2(b3, u3, mul2(b2, u2));
            a[i] = t[i]; ca[i] = ct;
        }
        {
            const float ct = ex2_approx(tS);
            const float du = tS - aS;
            const float x = caS * ct;
            const float dk = __fmaf_rn(gnegS, kf, ngdS);
            const float q2 = x * caS, q3 = x * ct;
            const float u2 = __fmaf_rn(q2, l2.x * du, q2) * (dk + gnegS);
            const float u3 = __fmaf_rn(q3, l3.x * du, q3) * ((dk + gnegS) + gnegS);
            g0S = __fmaf_rn(a3.x, u3, __fmaf_rn(a2.x, u2, __fmaf_rn(caS * caS * caS, dk, pgS)));
            g1S = __fmaf_rn(b3.x, u3, b2.x * u2);
            aS = tS; caS = ct;
        }
        kf += 3.f;
        if (jb >= j0) {
            float vA, vB;
            transpose(g0, g0S, vA, vB);
            if (RED) {
                if (st_a) atomicAdd(ga, vA);
                if (st_b) atomicAdd(gb, vB);
            } else {
                if (st_a) *ga = vA;
                if (st_b) *gb = vB;
            }
            ga += plane; gb += plane;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) pg[i] = g1[i];
        pgS = g1S;
    }
    } while (PERSIST && (ct += gridDim.x) < n_ct);        // CTA-task loop
}

// gcost += scratch, with the rows that never receive a "B" part (row 0 gets block row -1's; all rows are
// written by exactly one task in each buffer) -- plain elementwise add, fixed order => deterministic.
__global__ void __launch_bounds__(256)
head_bwd_combine_kernel(float* __restrict__ gcost, const float* __restrict__ scratch, size_t n4, size_t n) {
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n4) {
        float4 a = reinterpret_cast<float4*>(gcost)[i];
        const float4 s = __ldcs(reinterpret_cast<const float4*>(scratch) + i);
        a.x += s.x; a.y += s.y; a.z += s.z; a.w += s.w;
        reinterpret_cast<float4*>(gcost)[i] = a;
    }
    if (i == 0)
        for (size_t k = n4 * 4; k < n; ++k) gcost[k] += scratch[k];
}

}  // namespace rag
