// x3 disparity-head forward, "cube-root" kernel: ONE MUFU.EX2 per pixel per LOW-RES bin instead of one
// per full-resolution bin, and 7 (12 with the lambda correction) FP32 operations instead of 9 + 3 exp2.
//
// Along the disparity axis the reference (rag_model.py:40, F.interpolate trilinear x3) places full-res
// bin 3j+1 exactly on low-res bin j (lambda == 0, see below) and bins 3j+2, 3j+3 at lambda ~ 1/3, 2/3
// between low-res bins j and j+1.  With z the log2-domain exponent of a pixel at low-res bin j and
// c_j = 2^(z_j/3), the softmax terms of the three full-res bins centred on low-res bin j are
//     k = 3j   : 2^(z_{j-1}/3 + 2 z_j/3) = c_j^2 * c_{j-1}
//     k = 3j+1 : 2^(z_j)                  = c_j^2 * c_j
//     k = 3j+2 : 2^(2 z_j/3 + z_{j+1}/3) = c_j^2 * c_{j+1}
// so with ps_j = c_{j-1} + c_j, kj = 3j+1-kc:
//      sum_k p_k        +=  c_j^2 * (ps_j + c_{j+1})
//      sum_k (k-kc) p_k +=  c_j^2 * (kj*ps_j - c_{j-1} + (kj+1)*c_{j+1})
// ps_j and q_j = c_{j-1} - kj*ps_j are formed one step early (when c_j arrives), so a step needs only the
// new c_{j+1}: nothing rotates through three registers.  The clamped ends fall out of the same formula
// with c_{-1} := c_0 (k = 0 sits on bin 0) and c_{Dl} := c_{Dl-1}.  The FP32 pipe (32 lane-ops/clk per
// SM sub-partition, packed or not -- tools/ffma_mix.cu) is what bounds this kernel, not the SFU.
//
// PyTorch's fp32 lambdas are not exactly 1/3, 2/3 (UpSample.cuh:115-130: 0.33333588 / 0.66666794 at the
// top of a 64 -> 192 axis).  Ignoring that costs up to 1.4e-5 px at sigma = 1 and 8e-5 px at sigma = 5
// (measured in fp64), so the first-order term is applied: bin 3j+2 gets the factor
// 1 + ln2*d1_j*(z_{j+1}-z_j), bin 3j+3 the factor 1 + ln2*d2_j*(z_{j+1}-z_j), d = lambda_fp32 - q/3
// (|d| < 4e-6, the neglected second-order term is < 1e-9 relative).  +5 operations per step.
// The correction runs from the second window chunk on (d < 1e-6 below bin 48: the uncorrected first
// chunk costs < 4e-6 px at sigma = 1); x3r_step's CORR switches it per chunk.
//
// In the H and W axes the phase-1 rows/columns (dst = 3i+1) have lambda == 0 exactly for i >= 1
// (fma(fl(1/3), 3i+1.5, -0.5) rounds to i because the excess (i+0.5)*2^-25 is below half an ulp of i)
// and 1.5e-8 for i == 0, so the centre row/column of a 3x3 block is the low-res value itself: the
// bilinear stage needs 14 packed operations instead of 22.
//
// Everything else: centred 3x3 blocks, 4x32 blocks per CTA, 2-stage cp.async window of 16 low-res
// bins, lazily moved per-pixel reference exponent, fp32 group sums added once per chunk into fp32
// totals in shared memory, regression centred on D/2.
//
// Pixel pairs (p<row><col>):  Q0=(p00,p02) Q1=(p10,p12) Q2=(p20,p22) Q3=(p01,p21) S=p11.
#pragma once
#include <type_traits>

#include "disp_head_x3.cuh"

namespace rag {

// Lazy-rescale threshold in the z/3 domain: c <= 2^32, c^3 <= 2^96, 16-group sums of c^2*(k*ps + ...) <= 2^110:
// well inside fp32, and a pixel's reference then moves only when a bin beats it by more than 66 nats.  (With
// the 2^24 threshold of the older kernels the whole-warp rescale path ran so often on large-magnitude costs
// that the kernel took 0.39 ms instead of 0.17 ms at sigma = 20.)
constexpr float kX3rTau = 32.0f;
// When ANY pixel of the warp crosses kX3rTau the whole warp walks the rescale path anyway, so every pixel
// whose new bin beats its reference by more than kX3rPiggy re-anchors on that occasion: its next crossing
// moves further away at no extra cost (the reference lands exactly on a bin, so nothing is lost in precision).
constexpr float kX3rPiggy = 4.0f;

struct X3rPair {                          // per pixel pair
    float2 c[2];                          // ping-pong: c_j and (after the step) c_{j+1}
    float2 c2, ps, q;                     // c_j^2, c_{j-1}(1+e2) + c_j, c_{j-1} - kj*ps
    float2 S, T;                          // group sums: sum g, -sum (k-kc) g
};
struct X3rOne {
    float c[2], c2, ps, q, S, T;
};

// One group (the three full-res bins centred on low-res bin j).  `c` = c_j, `cn` receives c_{j+1}.
// nk1 = -(kj+1), nk3 = -(kj+3) = -k_{j+1}.
template <bool CORR>
__device__ __forceinline__ void x3r_step(const float2& c, float2& cn, float2& c2, float2& ps, float2& q, float2& S,
                                         float2& T, const float2& u_prev, const float2& u_new, float2 kap1,
                                         float2 kap2, float2 nk1, float2 nk3) {
    cn = ex2_2(u_new);
    float2 up = cn;
    float2 s2 = add2(c, cn);
    if (CORR) {
        const float2 du = fma2(u_prev, f2b(-1.f), u_new);
        up = fma2(cn, mul2(kap1, du), cn);
        s2 = fma2(c, mul2(kap2, du), s2);
    }
    S = fma2(c2, add2(ps, up), S);
    T = fma2(c2, fma2(nk1, up, q), T);
    c2 = mul2(cn, cn);
    ps = s2;
    q = fma2(nk3, s2, c);
}
template <bool CORR>
__device__ __forceinline__ void x3r_step(const float& c, float& cn, float& c2, float& ps, float& q, float& S, float& T,
                                         const float& u_prev, const float& u_new, float kap1, float kap2, float nk1,
                                         float nk3) {
    cn = ex2_approx(u_new);
    float up = cn;
    float s2 = c + cn;
    if (CORR) {
        const float du = u_new - u_prev;
        up = __fmaf_rn(cn, kap1 * du, cn);
        s2 = __fmaf_rn(c, kap2 * du, s2);
    }
    S = __fmaf_rn(c2, ps + up, S);
    T = __fmaf_rn(c2, __fmaf_rn(nk1, up, q), T);
    c2 = cn * cn;
    ps = s2;
    q = __fmaf_rn(nk3, s2, c);
}

// tiles: ceil(Wl/32) x ceil(Hl/WARPS) x B; 32*WARPS threads (a tile is WARPS block rows x 32 block columns); 1-D grid,
// one tile per CTA or a persistent grid (see the tile loop).
// smem: tile[STAGES][BINS][WARPS+2][kTCols] | float2 tot[18][NT] | float2 kap[Dl][2] ((k1,k1),(k2,k2))
// tot keeps (hi, lo) slots per total; only the hi words are accumulated, the lo words stay zero.
template <int WARPS, int MINB, int BINS, int STAGES>
__global__ void __launch_bounds__(32 * WARPS, MINB)
head_fwd_x3r_kernel(const float* __restrict__ cost, float* __restrict__ disp, float* __restrict__ stats,
                    int Dl, int Hl, int Wl, float scale, int nbx, int nby, int n_tl) {
    static_assert(BINS % 2 == 0, "two bins are staged per pass");
    constexpr int NT = 32 * WARPS, ROWS = WARPS + 2, HALF = NT / 2;
    static_assert(HALF >= ROWS * (kTCols / 4), "half a CTA stages one bin slab per pass");
    static_assert(NT >= BINS * ROWS, "one thread per window row for the edge patches");
    extern __shared__ __align__(16) float x3r_smem[];
    constexpr int kStageFloats = BINS * ROWS * kTCols;
    constexpr int kBinFloats = ROWS * kTCols;
    const int D = 3 * Dl, W = 3 * Wl;
    float* tile = x3r_smem;
    float2* tot = reinterpret_cast<float2*>(x3r_smem + STAGES * kStageFloats);   // [18][128]
    float2* kap = tot + 18 * NT;                                                   // [Dl][2]
    int tid = threadIdx.x;
    asm volatile("" : "+r"(tid));     // one read: the compiler otherwise re-reads SR_TID (27 S2R per chunk of bins) wherever it needs a thread index
    const int lane = tid & 31, warp = tid >> 5;
    // kappa_q(j) = 3 ln2 (lambda_fp32(3j+1+q) - q/3), q = 1, 2: the 3 converts du (z/3 domain) to dz.
    // lambda - fl(q/3) is exact in fp32 (Sterbenz); fl(1/3) - 1/3 = 2^-25/3, fl(2/3) - 2/3 = 2^-24/3.
    // Once per CTA; published by the first chunk barrier of the first tile.
    for (int j = tid; j < Dl; j += NT) {
        float k12[2];
#pragma unroll
        for (int q = 1; q <= 2; ++q) {
            int t0, t1;
            float l0, l1;
            src_index<true>(scale, min(3 * j + 1 + q, D - 1), Dl, t0, t1, l0, l1);
            const float third = q == 1 ? 0.333333343267440796f : 0.666666686534881592f;
            const float resid = q == 1 ? 9.934107e-9f : 1.9868214e-8f;
            const float d = (t1 > t0) ? (l1 - third) + resid : 0.f;   // clamped top bin: no interval
            k12[q - 1] = 2.0794415416798357f * d;
        }
        kap[2 * j + 0] = f2b(k12[0]);
        kap[2 * j + 1] = f2b(k12[1]);
    }
    // tiles (32 block columns x WARPS block rows x image) tl = (b * nby + by) * nbx + bx; CTA blockIdx.x works on
    // tl = blockIdx.x, blockIdx.x + gridDim.x, ...: one tile per CTA by default, a persistent grid of a few CTAs per SM
    // (resident at once: RAG_HEAD_FWD_SHARED, rag_b200.pipeline) when the kernel shares the SMs with a volume kernel
    for (int tl = blockIdx.x; tl < n_tl; tl += gridDim.x) {
    const int tq = tl / nbx;
    const int b = tq / nby;
    const int C0 = (tl - tq * nbx) * 32, R0 = (tq - b * nby) * WARPS;
    const int T0 = C0 - 4;
    const size_t plane = (size_t)Hl * Wl;
    const float* base = cost + (size_t)b * Dl * plane;
    const int Wv = Wl >> 2;
    const int n_chunks = (Dl + BINS - 1) / BINS;
    const bool patch_l = C0 == 0;
    const bool patch_r = (Wl - T0) <= 36;
    const int pr = Wl - T0;

    // window staging: one bin slab = ROWS rows x 10 vectors.  The first half of the CTA copies the even bins
    // of a chunk, the second half the odd ones; a thread's (row, vector) and so its source offset inside
    // a bin plane never change.
    const int st_half = tid >= HALF ? 1 : 0, st_u = tid - st_half * HALF;
    const bool st_on = st_u < ROWS * (kTCols / 4);
    const int st_row = st_u / (kTCols / 4), st_vec = st_u % (kTCols / 4);
    const int st_soff = st_half * kBinFloats + st_row * kTCols + st_vec * 4;
    const float* st_src = base + (size_t)min(max(R0 - 1 + st_row, 0), Hl - 1) * Wl + 4 * min(max((T0 >> 2) + st_vec, 0), Wv - 1);
    auto issue_chunk = [&](int ch) {
        if (ch < n_chunks && st_on) {
            float* dst = tile + (ch % STAGES) * kStageFloats + st_soff;
#pragma unroll
            for (int q = 0; q < BINS / 2; ++q) {
                const int gj = min(ch * BINS + 2 * q + st_half, Dl - 1);
                __pipeline_memcpy_async(dst + 2 * q * kBinFloats, st_src + (size_t)gj * plane, 16);
            }
        }
        __pipeline_commit();
    };
    issue_chunk(0);
    if (STAGES > 2) issue_chunk(1);
    float2* mytot = tot + tid;
#pragma unroll
    for (int s = 0; s < 18; ++s) mytot[s * NT] = f2b(0.f);

    const int r_raw = R0 + warp, c_raw = C0 + lane;
    const bool active = r_raw < Hl && c_raw < Wl;
    const int r = min(r_raw, Hl - 1), c = min(c_raw, Wl - 1);
    constexpr float kS3 = kX3NegLog2e / 3.0f;            // exponents are produced as z/3 = -log2e*v/3
    float hs0[3], hs1[3], wl0[3], wl1[3];
#pragma unroll
    for (int i = 0; i < 3; i += 2) {                     // phases 0 and 2; phase 1 is the low-res sample itself
        int i0, i1;
        float l0, l1;
        src_index<true>(scale, 3 * r + i, Hl, i0, i1, l0, l1);
        hs0[i] = l0 * kS3; hs1[i] = l1 * kS3;
        src_index<true>(scale, 3 * c + i, Wl, i0, i1, wl0[i], wl1[i]);
    }
    const int org = (r - R0) * kTCols + (c - C0 + 3);
    // col 0 = wl0[0]*v0 + wl1[0]*v1, col 2 = wl0[2]*v1 + wl1[2]*v2  ->  (col0,col2) = wM*v1 + wO*(v0,v2)
    const float2 wO = f2(wl0[0], wl1[2]), wM = f2(wl1[0], wl0[2]);
    // centre column: row 0 = hs0[0]*v1[0] + hs1[0]*v1[1], row 2 = hs0[2]*v1[1] + hs1[2]*v1[2]
    const float2 hO = f2(hs0[0], hs1[2]), hM = f2(hs1[0], hs0[2]);
    const float2 h00 = f2b(hs0[0]), h10 = f2b(hs1[0]), h02 = f2b(hs0[2]), h12 = f2b(hs1[2]);
    const float2 s3b = f2b(kS3);

    float2 mneg[4], ua[4], ub[4];     // -m/3; ping-pong relative exponents (z - m)/3 of low-res bins j, j+1
    float mnegS = 0.f, uaS = 0.f, ubS = 0.f;
    X3rPair st[4];
    X3rOne so = {{1.f, 1.f}, 1.f, 2.f, 0.f, 0.f, 0.f};
    const float kc = 0.5f * (float)D;
    float nk = kc - 1.f;              // -kj = -(3j + 1 - kc)

    // (z - m)/3 of the nine pixels at the low-res bin whose window slab starts at p
    auto blend = [&](const float* p, const float2 (&mn)[4], float mnS, float2 (&o)[4], float& oS) {
        // operands are either natural pairs of two separate loads ((v0,v2) of a row, (v1 row0, v1 row2)) or
        // scalars broadcast by the instruction, so no pair has to be assembled with MOVs
        float2 xc[3];
#pragma unroll
        for (int rr = 0; rr < 3; ++rr) {
            const float2 v02 = f2(p[rr * kTCols + 0], p[rr * kTCols + 2]);
            xc[rr] = fma2(wM, f2b(p[rr * kTCols + 1]), mul2(wO, v02));      // (col 0, col 2) of window row rr
        }
        const float2 v1e = f2(p[0 * kTCols + 1], p[2 * kTCols + 1]);
        const float v1c = p[1 * kTCols + 1];
        o[0] = fma2(h00, xc[0], fma2(h10, xc[1], mn[0]));
        o[1] = fma2(s3b, xc[1], mn[1]);
        o[2] = fma2(h02, xc[1], fma2(h12, xc[2], mn[2]));
        o[3] = fma2(hM, f2b(v1c), fma2(hO, v1e, mn[3]));
        oS = __fmaf_rn(kS3, v1c, mnS);
    };
    // group sums -> totals: the chunk sums are simply added in fp32 (at most ~1.5 ulp on top of the in-chunk rounding).
    auto fold = [&]() {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            mytot[(4 * i + 0) * NT] = add2(mytot[(4 * i + 0) * NT], st[i].S);
            mytot[(4 * i + 2) * NT] = add2(mytot[(4 * i + 2) * NT], st[i].T);
            st[i].S = f2b(0.f); st[i].T = f2b(0.f);
        }
        float2 d = mytot[16 * NT], n = mytot[17 * NT];
        d.x += so.S; n.x += so.T;
        mytot[16 * NT] = d; mytot[17 * NT] = n;
        so.S = 0.f; so.T = 0.f;
    };
    // rare path: the new bin's exponent `t` exceeds the pixel's reference by more than kX3rTau.  The
    // reference moves onto that bin: totals scale by 2^(-3t), the carried c-linear terms by 2^(-t).
    // `cur` = which half of the c ping-pong holds c_j.
    auto rescale = [&](auto cur_tag, float2 (&t)[4], float& tS, float2 (&a)[4], float& aS) {
        constexpr int cur = decltype(cur_tag)::value;
        // the running group sums (registers) and the chunk totals (shared memory; hi words only, the lo words are
        // zero) are both scaled in place -- no fold, so an event costs ~160 instead of ~270 instructions
        auto fix = [&](float& tt, float& aa, float& mn, float& cc, float& c2, float& ps, float& q, float& gs, float& gt,
                       int slot, bool hi_lane) {
            if (tt > kX3rPiggy) {
                const float f = ex2_approx(-tt), f3 = ex2_approx(-3.f * tt);
#pragma unroll
                for (int s = 0; s < 4; s += 2) {
                    float2 v = mytot[(slot + s) * NT];
                    if (hi_lane) v.y *= f3; else v.x *= f3;
                    mytot[(slot + s) * NT] = v;
                }
                gs *= f3; gt *= f3;
                cc *= f; ps *= f; q *= f; c2 = cc * cc;
                mn -= tt; aa -= tt; tt = 0.f;
            }
        };
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            fix(t[i].x, a[i].x, mneg[i].x, st[i].c[cur].x, st[i].c2.x, st[i].ps.x, st[i].q.x, st[i].S.x, st[i].T.x, 4 * i, false);
            fix(t[i].y, a[i].y, mneg[i].y, st[i].c[cur].y, st[i].c2.y, st[i].ps.y, st[i].q.y, st[i].S.y, st[i].T.y, 4 * i, true);
        }
        if (tS > kX3rPiggy) {
            const float f = ex2_approx(-tS), f3 = ex2_approx(-3.f * tS);
            float2 d = mytot[16 * NT], n = mytot[17 * NT];
            d.x *= f3; d.y *= f3; n.x *= f3; n.y *= f3;
            mytot[16 * NT] = d; mytot[17 * NT] = n;
            so.S *= f3; so.T *= f3;
            so.c[cur] *= f; so.ps *= f; so.q *= f; so.c2 = so.c[cur] * so.c[cur];
            mnegS -= tS; aS -= tS; tS = 0.f;
        }
    };
    auto maxof = [](const float2 (&t)[4], float tS) {
        return fmaxf(fmaxf(fmaxf(fmaxf(t[0].x, t[0].y), fmaxf(t[1].x, t[1].y)),
                           fmaxf(fmaxf(t[2].x, t[2].y), fmaxf(t[3].x, t[3].y))), tS);
    };
    // group j: c_j sits in half `cur` of the ping-pong, c_{j+1} goes to the other half
    auto group = [&](auto cur_tag, auto corr_tag, const float2 (&up)[4], float upS, const float2 (&un)[4], float unS,
                     float2 k1, float2 k2) {
        constexpr int cur = decltype(cur_tag)::value;
        constexpr bool corr = decltype(corr_tag)::value;
        const float nk1 = nk - 1.f, nk3 = nk - 3.f;
        const float2 nk1b = f2b(nk1), nk3b = f2b(nk3);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            x3r_step<corr>(st[i].c[cur], st[i].c[cur ^ 1], st[i].c2, st[i].ps, st[i].q, st[i].S, st[i].T, up[i], un[i], k1, k2, nk1b, nk3b);
        x3r_step<corr>(so.c[cur], so.c[cur ^ 1], so.c2, so.ps, so.q, so.S, so.T, upS, unS, k1.x, k2.x, nk1, nk3);
        nk = nk3;
    };
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    // the steps of one chunk: two groups per trip, exponent registers (ua -> ub -> ua) and c halves ping-pong.
    // A pixel running away from its reference (rare) BREAKS out of the hot loop, is handled below it and
    // the loop is re-entered, so that the hot loop is straight-line code with fall-through exits only.
    auto hot = [&](float mx) { return __any_sync(0xffffffffu, mx > kX3rTau); };
    auto run_chunk = [&](auto corr_tag, const float* p, int n_it, const float2* kp) {
        for (;;) {
            int rare = 0;
            float mx = 0.f;
            for (; n_it >= 2; n_it -= 2) {
                blend(p, mneg, mnegS, ub, ubS);
                mx = maxof(ub, ubS);
                if (hot(mx)) { rare = 1; break; }
                group(I0{}, corr_tag, ua, uaS, ub, ubS, kp[0], kp[1]);
                blend(p + kBinFloats, mneg, mnegS, ua, uaS);
                mx = maxof(ua, uaS);
                if (hot(mx)) { rare = 2; break; }
                group(I1{}, corr_tag, ub, ubS, ua, uaS, kp[2], kp[3]);
                p += 2 * kBinFloats;
                kp += 4;
            }
            if (rare == 0) break;
            if (rare == 1) {
                rescale(I0{}, ub, ubS, ua, uaS);
                group(I0{}, corr_tag, ua, uaS, ub, ubS, kp[0], kp[1]);
                blend(p + kBinFloats, mneg, mnegS, ua, uaS);
                if (hot(maxof(ua, uaS))) rescale(I1{}, ua, uaS, ub, ubS);
            } else {
                rescale(I1{}, ua, uaS, ub, ubS);
            }
            group(I1{}, corr_tag, ub, ubS, ua, uaS, kp[2], kp[3]);
            p += 2 * kBinFloats;
            kp += 4;
            n_it -= 2;
        }
        if (n_it == 1) {
            blend(p, mneg, mnegS, ub, ubS);
            if (hot(maxof(ub, ubS))) rescale(I0{}, ub, ubS, ua, uaS);
            group(I0{}, corr_tag, ua, uaS, ub, ubS, kp[0], kp[1]);
#pragma unroll
            for (int i = 0; i < 4; ++i) { ua[i] = ub[i]; st[i].c[0] = st[i].c[1]; }
            uaS = ubS; so.c[0] = so.c[1];
        }
    };

    for (int ch = 0; ch < n_chunks; ++ch) {
        issue_chunk(ch + STAGES - 1);
        __pipeline_wait_prior(STAGES - 1);
        __syncthreads();
        float* stw = tile + (ch % STAGES) * kStageFloats;
        if (patch_l || patch_r) {
            if (tid < BINS * ROWS) {
                float* rowp = stw + tid * kTCols;
                if (patch_l) rowp[3] = rowp[4];
                if (patch_r) rowp[pr] = rowp[pr - 1];
            }
            __syncthreads();
        }
        const int jbeg = ch * BINS, jend = min(jbeg + BINS, Dl);
        const float* p = stw + org;
        if (ch == 0) {
            const float2 z4[4] = {f2b(0.f), f2b(0.f), f2b(0.f), f2b(0.f)};
            blend(p, z4, 0.f, ub, ubS);          // plain z/3 of low-res bin 0 = the reference exponents
            // c_0 = 2^0; c_{-1} := c_0, so ps_0 = 2 and q_0 = c_{-1} - k_0 * ps_0
            const float q0 = __fmaf_rn(nk, 2.f, 1.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                mneg[i] = f2(-ub[i].x, -ub[i].y);
                ua[i] = f2b(0.f);
                st[i].c[0] = f2b(1.f); st[i].c[1] = f2b(1.f); st[i].c2 = f2b(1.f);
                st[i].ps = f2b(2.f); st[i].q = f2b(q0);
                st[i].S = f2b(0.f); st[i].T = f2b(0.f);
            }
            mnegS = -ubS; uaS = 0.f;
            so.c[0] = 1.f; so.c[1] = 1.f; so.c2 = 1.f; so.ps = 2.f; so.q = q0; so.S = 0.f; so.T = 0.f;
            p += kBinFloats;
        }
        const int n_it = jend - max(jbeg, 1);
        const float2* kp = kap + 2 * (max(jbeg, 1) - 1);
        if (ch > 0) run_chunk(std::true_type{}, p, n_it, kp);
        else run_chunk(std::false_type{}, p, n_it, kp);
        fold();
        __syncthreads();
    }
    // last group (j = Dl-1): k = 3Dl-1 clamps onto low-res bin Dl-1, i.e. c_{Dl} := c_{Dl-1}, du = 0
    {
        const float nk1 = nk - 1.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 cc = st[i].c[0];
            st[i].S = mul2(st[i].c2, add2(st[i].ps, cc));
            st[i].T = mul2(st[i].c2, fma2(f2b(nk1), cc, st[i].q));
        }
        so.S = so.c2 * (so.ps + so.c[0]);
        so.T = so.c2 * __fmaf_rn(nk1, so.c[0], so.q);
    }
    fold();
    if (active) {
    const size_t img = (size_t)3 * Hl * W;
    float* dp = disp + (size_t)b * img + (size_t)(3 * r) * W + 3 * c;
    float* sp = stats ? stats + (size_t)b * 2 * img + (size_t)(3 * r) * W + 3 * c : nullptr;
    // totals: d = sum 2^(z_k - m), n = -sum (k - kc) 2^(z_k - m)
    auto emit = [&](int ph, int pw, float dhi, float dlo, float nhi, float nlo, float mn) {
        const int o = ph * W + pw;
        const float inv = __frcp_rn(dhi + dlo);
        const float q = nhi * inv;
        const float rr2 = __fmaf_rn(-q, dhi, nhi) + (nlo - q * dlo);
        dp[o] = kc - (q + rr2 * inv);
        if (sp) {
            // reference exponent in the z domain: m = -3*mn = mhi + mlo; the rounding residue mlo is
            // folded into the stored normaliser so that 2^(z - mhi) * inv' == 2^(z - m) * inv
            const float mhi = -3.f * mn;
            const float mlo = __fmaf_rn(-3.f, mn, -mhi);
            sp[o] = mhi;
            sp[img + o] = inv * ex2_approx(-mlo);
        }
    };
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 dhi = mytot[(4 * i + 0) * NT], dlo = mytot[(4 * i + 1) * NT];
        const float2 nhi = mytot[(4 * i + 2) * NT], nlo = mytot[(4 * i + 3) * NT];
        if (i < 3) {
            emit(i, 0, dhi.x, dlo.x, nhi.x, nlo.x, mneg[i].x);
            emit(i, 2, dhi.y, dlo.y, nhi.y, nlo.y, mneg[i].y);
        } else {
            emit(0, 1, dhi.x, dlo.x, nhi.x, nlo.x, mneg[i].x);
            emit(2, 1, dhi.y, dlo.y, nhi.y, nlo.y, mneg[i].y);
        }
    }
    {
        const float2 d = mytot[16 * NT], n = mytot[17 * NT];
        emit(1, 1, d.x, d.y, n.x, n.y, mnegS);
    }
    }   // active
    }   // tile loop
}

}  // namespace rag
