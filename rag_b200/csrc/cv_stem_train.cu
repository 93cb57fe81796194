// Backward of the fused cost volume + stem3d0 layer WITHOUT the volume or its gradient (SURVEY.md section 8f rank 1,
// "and its mirror in backward").  Reference: the autograd of src/models/rag_model.py:375-383 followed by
// `self.stem3d0[i](cost)` = ConvBR_3d(2C -> O, 3x3x3, pad 1) + BatchNorm3d + ReLU (rag_model.py:234,341,
// src/automl/operations_3d.py:31-47), in train() (batch statistics) or eval() (running statistics).
//
// The forward is z[o,d,h,w] = sum_{c,kd,kh,kw} W[o,ci,kd,kh,kw] V[ci,d+kd-1,h+kh-1,w+kw-1] with the volume V a masked /
// shifted broadcast of the two feature maps: V[c,d',h',w'] = x[c,h',w'] [w'>=d'], V[C+c,d',h',w'] = y[c,h',w'-d'] [w'>=d'].
// So the gradient w.r.t. x, y and W only needs, per output row (b,o,h), a few SUMS OVER d of the upstream gradient gz:
//     Tw[kd,kw][w] = sum_d gz[d,w] [0 <= d+kd-1 < Df] [d+kd-1 <= w+kw-1]        (triangular prefix sums of a column)
//     S[kdc,kwc][e] = sum_d gz[d,e+d] over the diagonal e = w-d, with d >= 1 if kdc == 0, d <= Df-2 if kdc == 2,
//                     w <= Wf-2 if kwc == 1                                        (diagonal sums, 6 classes)
// and then 2-D contractions (h' = h+kh-1):
//     gx[c,h',w'] = sum_{o,kd,kh,kw} W[o,  c,kd,kh,kw] Tw[kd,kw][o,h,w'-kw+1]
//     gy[c,h',u ] = sum_{o,kd,kh,kw} W[o,C+c,kd,kh,kw] S[kd,kw==2][o,h,u+kd-kw]
//     gW[o,  c,kd,kh,kw] = sum_{b,h,w'} x[c,h',w'] Tw[kd,kw][o,h,w'-kw+1]
//     gW[o,C+c,kd,kh,kw] = sum_{b,h,u } y[c,h',u ] S[kd,kw==2][o,h,u+kd-kw]
// (the fp64 prototype of this algebra is checked against the reference's autograd through the materialised volume in the
// CPU test-suite: stem_backward_volume_free_f64, tests/test_oracle_golden.py).  gz itself is never stored either: the maps
// kernel rebuilds it on the fly from the upstream gradient g of the layer OUTPUT and the convolution output z, with the
// BatchNorm constants and the ReLU decision of bn3d.cu.  The BatchNorm backward needs z, not only the output, so instead of
// keeping a second [B,O,Df,Hf,Wf] tensor alive the host side RECOMPUTES z with the forward kernel into a temporary.
// Backward passes over g and z: ONE for the two BatchNorm sums (bn3d.cu), ONE for the maps (bwd_maps); everything after that
// works on 2-D maps (15/Df of the tensor size).
// CV-2's descending-d summation order does not apply here: the reference's own gz comes out of cuDNN, so the bar is
// the 1e-5 max-norm of the other floating-point rows, not bit equality.
#include <algorithm>

#include "common.cuh"

namespace rag {

constexpr int kStC = 12;          // feature channels (the fused stem is specialised for the reference's C = 12)
constexpr int kStWC = 128;        // column chunk of the contraction kernels
constexpr int kStQ = 3 * kStC;    // (c, kh) pairs

// ---- the d-sums of gz -----------------------------------------------------------------------------------------------
// grid (Hf, O, B); blockDim = roundup32(Wf + 4): thread t owns column w = t (t < Wf) and diagonal e = t - 2 (t < Wf + 2).
// consts [O][7] = (a, m1, m2, scale, shift, mean, rstd).  tmap [B,O,Hf,9,Wf]; umap [B,O,Hf,6,Wf+4] (entry e+2; the last two are 0).
// U = rows per batch (divides Df: no row predicates in the loop).  smem: 2 x U rows of gz for the column -> diagonal
// exchange | 5 x Wf prefix snapshots (column w needs its prefix sum at d = w-2 .. w+2: written by the five rows that pass
// through it -- a rarely taken predicated store instead of five live registers).
template <int U>
__global__ void __launch_bounds__(1024)
stem_bwd_maps_kernel(const float* __restrict__ g, const float* __restrict__ out, const float* __restrict__ consts,
                     float* __restrict__ tmap, float* __restrict__ umap, int O, int Df, int Hf, int Wf) {
    extern __shared__ float stm_smem[];                    // [2][U][Wf] | [5][Wf]
    float* snaps = stm_smem + 2 * U * Wf;
    const int h = blockIdx.x, o = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const int w = tid, e = tid - 2;
    const bool col = w < Wf, diag = tid < Wf + 2;
    const size_t plane = (size_t)Hf * Wf;
    const size_t base = ((size_t)(b * O + o) * Df) * plane + (size_t)h * Wf + min(w, Wf - 1);   // threads past the row re-read its last column
    const float* pg = g + base;
    const float* po = out + base;
    const float a = __ldg(consts + 7 * o), m1 = __ldg(consts + 7 * o + 1), m2 = __ldg(consts + 7 * o + 2);
    const float sc = __ldg(consts + 7 * o + 3), sh = __ldg(consts + 7 * o + 4), mu = __ldg(consts + 7 * o + 5), rs = __ldg(consts + 7 * o + 6);
    if (col) {
#pragma unroll
        for (int k = 0; k < 5; ++k) snaps[k * Wf + w] = 0.f;
    }
    float run = 0.f, first = 0.f, glast = 0.f;
    // diagonal: ONE running sum + the (at most one each) elements a tap class excludes: d = 0, d = Df-1, w = Wf-1
    float Sall = 0.f, f0 = 0.f, fl = 0.f, fc = 0.f;
    const int d_c = Wf - 1 - e;                             // the d at which diagonal e crosses the last column
    const int wm2 = w - 2;
    int buf = 0;
    for (int d0 = 0; d0 < Df; d0 += U) {
        float gv[U], ov[U];
#pragma unroll
        for (int i = 0; i < U; ++i) {
            gv[i] = ld_stream(pg + (size_t)i * plane);
            ov[i] = ld_stream(po + (size_t)i * plane);
        }
        pg += (size_t)U * plane;
        po += (size_t)U * plane;
        float* rowbuf = stm_smem + buf * U * Wf;
        float gz[U];
#pragma unroll
        for (int i = 0; i < U; ++i) {
            const float gp = __fmaf_rn(ov[i], sc, sh) > 0.f ? gv[i] : 0.f;   // the forward's own ReLU decision, bit for bit
            const float zh = (ov[i] - mu) * rs;              // needed everywhere in train mode: the -a (m1 + zh m2) term does not stop at the ReLU
            gz[i] = a * (gp - m1 - zh * m2);
        }
        if (col) {
#pragma unroll
            for (int i = 0; i < U; ++i) {
                run += gz[i];
                rowbuf[i * Wf + w] = gz[i];
                const unsigned k = (unsigned)(d0 + i - wm2);  // the five prefix snapshots a column needs sit at d = w-2 .. w+2
                if (k < 5u) snaps[k * Wf + w] = run;
            }
            if (d0 == 0) first = gz[0];
            glast = gz[U - 1];
        }
        __syncthreads();
        if (diag) {
#pragma unroll
            for (int i = 0; i < U; ++i) {
                const int dd = d0 + i, cc = e + dd;
                if ((unsigned)cc < (unsigned)Wf) {
                    const float v = rowbuf[i * Wf + cc];
                    Sall += v;
                    f0 = dd == 0 ? v : f0;
                    fl = dd == Df - 1 ? v : fl;
                    fc = dd == d_c ? v : fc;
                }
            }
        }
        buf ^= 1;
    }
    float S[6];
    {
        // classes (kd class, kw == 2): kd 0 drops d = 0, kd 2 drops d = Df-1, kw == 2 drops w = Wf-1; an element that is both
        // (d = 0 or Df-1) AND in the last column must be dropped once
        const bool c0 = d_c == 0, cl = d_c == Df - 1;       // the last-column element IS the d = 0 / d = Df-1 element
        S[0] = Sall - f0;
        S[1] = Sall - f0 - (c0 ? 0.f : fc);
        S[2] = Sall;
        S[3] = Sall - fc;
        S[4] = Sall - fl;
        S[5] = Sall - fl - (cl ? 0.f : fc);
    }
    const size_t row = (size_t)(b * O + o) * Hf + h;
    if (col) {
        const float total = run, last2 = run - glast;
        auto P = [&](int j) -> float {                  // prefix sum of the column up to bin j (inclusive)
            if (j >= Df - 1) return total;
            if (j == Df - 2) return last2;
            if (j == 0) return first;
            return snaps[(j - wm2) * Wf + w];           // j in [w-2, w+2] (own writes: no barrier needed)
        };
        float* tp = tmap + row * 9 * Wf + w;
#pragma unroll
        for (int kd = 0; kd < 3; ++kd)
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int wp = w + kw - 1;                   // input column this output column reads through tap kw
                float t = 0.f;
                if (wp >= 0 && wp < Wf) {
                    const int upper = min(Df - 1, min(Df - 1, wp) - kd + 1);
                    const int lower = kd == 0 ? 1 : 0;
                    if (upper >= lower) t = P(upper) - (lower == 1 ? first : 0.f);
                }
                tp[(size_t)(kd * 3 + kw) * Wf] = t;
            }
    }
    if (tid < Wf + 4) {
        float* up = umap + row * 6 * (Wf + 4) + tid;
#pragma unroll
        for (int c6 = 0; c6 < 6; ++c6) up[(size_t)c6 * (Wf + 4)] = diag ? S[c6] : 0.f;
    }
}

// ---- gx, gy: out[c][h'][w'] = sum_{kh} sum_{r=(o,kd,kw)} W[o,side*C+c,kd,kh,kw] * M_r[h'-kh+1][shifted w'] --------------
// A CTA owns kStTH output rows x 128 columns of one (b, side) and walks the kStTH + 2 map rows that feed them: each map
// row is staged ONCE (pre-shifted per tap so that every read is an aligned LDS.128) and used for its three kh taps.
// 256 threads = 2 halves of the r range x 4 channel groups (3 channels) x 32 column quads; the halves are added through
// shared memory at the end.  grid (ceil(Wf/128), ceil(Hf/kStTH), 2*B): blockIdx.z = 2*b + side.
// smem: Ms[R][128] | Ws[3][R][4][4]   (R = 9*O; the reduction buffer aliases Ms)
constexpr int kStTH = 4;
__global__ void __launch_bounds__(256)
stem_bwd_inputs_kernel(const float* __restrict__ tmap, const float* __restrict__ umap, const float* __restrict__ wgt,
                       float* __restrict__ gx, float* __restrict__ gy, int O, int Hf, int Wf) {
    extern __shared__ __align__(16) float sti_smem[];
    const int R = 9 * O;
    float* Ms = sti_smem;
    float* Ws = Ms + (size_t)R * kStWC;
    const int w0 = blockIdx.x * kStWC, hp0 = blockIdx.y * kStTH, b = blockIdx.z >> 1, side = blockIdx.z & 1, tid = threadIdx.x;
    const int half = tid >> 7, tc = (tid >> 5) & 3, tj = tid & 31, warp = tid >> 5, lane = tid & 31;
    float acc[kStTH][3][4];
#pragma unroll
    for (int t = 0; t < kStTH; ++t)
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[t][i][j] = 0.f;
    for (int i = tid; i < 3 * R * 16; i += 256) {            // Ws[kh][r][channel group][3 channels + pad]: one LDS.128 per tap
        const int kh = i / (R * 16), rc = i - kh * R * 16;
        const int r = rc >> 4, cg = (rc >> 2) & 3, ci = rc & 3;
        const int o = r / 9, kd = (r % 9) / 3, kw = r % 3;
        Ws[i] = ci < 3 ? __ldg(wgt + ((((size_t)o * 2 * kStC + side * kStC + 3 * cg + ci) * 3 + kd) * 3 + kh) * 3 + kw) : 0.f;
    }
    const int r_beg = half * ((R + 1) >> 1), r_end = half ? R : ((R + 1) >> 1);
    // map row h = hp0 - 1 + hh feeds output rows h-1, h, h+1 through kh = 0, 1, 2: tile-local output row hh + kh - 2.  The
    // hh loop is unrolled so that the accumulator index is a compile-time constant (a run-time index would turn the 12 FMAs
    // of a tap into 48 predicated ones).
#pragma unroll
    for (int hh = 0; hh < kStTH + 2; ++hh) {
        const int h = hp0 - 1 + hh;
        if (h < 0 || h >= Hf) continue;                      // block-uniform
        __syncthreads();
        for (int r = warp; r < R; r += 8) {                  // a warp stages whole rows: coalesced, no div/mod per element
            const int o = r / 9, kd = (r % 9) / 3, kw = r % 3;
            const size_t row = (size_t)(b * O + o) * Hf + h;
            const float* src;
            int shift, lim;
            if (side == 0) { src = tmap + (row * 9 + kd * 3 + kw) * Wf; shift = 1 - kw; lim = Wf; }          // Tw indexed by the OUTPUT column
            else { src = umap + (row * 6 + kd * 2 + (kw == 2 ? 1 : 0)) * (Wf + 4); shift = kd - kw + 2; lim = Wf + 4; }   // diagonal e = u + kd - kw at e + 2
#pragma unroll
            for (int k = 0; k < kStWC / 32; ++k) {
                const int j = lane + 32 * k, idx = w0 + j + shift;
                Ms[r * kStWC + j] = (idx >= 0 && idx < lim && w0 + j < Wf) ? __ldg(src + idx) : 0.f;
            }
        }
        __syncthreads();
        for (int r = r_beg; r < r_end; ++r) {
            const float4 t = *reinterpret_cast<const float4*>(Ms + (size_t)r * kStWC + 4 * tj);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
                constexpr int dummy = 0; (void)dummy;
                const int tl = hh + kh - 2;                  // compile-time after unrolling
                if (tl < 0 || tl >= kStTH) continue;
                const float4 wv = *reinterpret_cast<const float4*>(Ws + (((size_t)kh * R + r) * 4 + tc) * 4);   // 3 channels + pad
                acc[tl][0][0] = __fmaf_rn(wv.x, t.x, acc[tl][0][0]); acc[tl][0][1] = __fmaf_rn(wv.x, t.y, acc[tl][0][1]);
                acc[tl][0][2] = __fmaf_rn(wv.x, t.z, acc[tl][0][2]); acc[tl][0][3] = __fmaf_rn(wv.x, t.w, acc[tl][0][3]);
                acc[tl][1][0] = __fmaf_rn(wv.y, t.x, acc[tl][1][0]); acc[tl][1][1] = __fmaf_rn(wv.y, t.y, acc[tl][1][1]);
                acc[tl][1][2] = __fmaf_rn(wv.y, t.z, acc[tl][1][2]); acc[tl][1][3] = __fmaf_rn(wv.y, t.w, acc[tl][1][3]);
                acc[tl][2][0] = __fmaf_rn(wv.z, t.x, acc[tl][2][0]); acc[tl][2][1] = __fmaf_rn(wv.z, t.y, acc[tl][2][1]);
                acc[tl][2][2] = __fmaf_rn(wv.z, t.z, acc[tl][2][2]); acc[tl][2][3] = __fmaf_rn(wv.z, t.w, acc[tl][2][3]);
            }
        }
    }
    // add the two halves of the r range (fixed order: half 0 + half 1) and store
    __syncthreads();
    float* red = Ms;                                         // [128 threads][48]
    if (half == 1) {
#pragma unroll
        for (int t = 0; t < kStTH; ++t)
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) red[((t * 3 + i) * 4 + j) * 128 + (tid & 127)] = acc[t][i][j];
    }
    __syncthreads();
    const int wq = w0 + 4 * tj;
    if (half == 0 && wq < Wf) {                              // Wf % 4 == 0: a quad is inside or outside as a whole
#pragma unroll
        for (int t = 0; t < kStTH; ++t) {
            const int hp = hp0 + t;
            if (hp >= Hf) continue;
            float* dst = (side == 0 ? gx : gy) + ((size_t)(b * kStC + 3 * tc) * Hf + hp) * Wf + wq;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                float4 v;
                v.x = acc[t][i][0] + red[((t * 3 + i) * 4 + 0) * 128 + tid];
                v.y = acc[t][i][1] + red[((t * 3 + i) * 4 + 1) * 128 + tid];
                v.z = acc[t][i][2] + red[((t * 3 + i) * 4 + 2) * 128 + tid];
                v.w = acc[t][i][3] + red[((t * 3 + i) * 4 + 3) * 128 + tid];
                *reinterpret_cast<float4*>(dst + (size_t)i * Hf * Wf) = v;
            }
        }
    }
}

// ---- gW partials: part[b,h,side][r=(o,kd,kw)][q=(c,kh)] = sum_w M_r[h][shifted w] * F[c][h+kh-1][w] -----------------
// grid (Hf, 2*B); threads: (Rp/4) x 9 register tiles of 4 x 4, Rp = 9*O rounded up to 4.
// smem: Ms[Rp][132] | Fs[36][132]: rows padded by 4 floats so that the 4-9 DIFFERENT rows the threads of a warp read at
// the same column land in different bank groups (a 512-byte stride would put them all on the same banks).
constexpr int kStWS = kStWC + 4;
__global__ void __launch_bounds__(1024)
stem_bwd_weight_kernel(const float* __restrict__ tmap, const float* __restrict__ umap, const float* __restrict__ x,
                       const float* __restrict__ y, float* __restrict__ part, int O, int Hf, int Wf) {
    extern __shared__ __align__(16) float stw_smem[];
    const int R = 9 * O, Rp = (R + 3) & ~3;
    float* Ms = stw_smem;
    float* Fs = Ms + (size_t)Rp * kStWS;
    const int h = blockIdx.x, b = blockIdx.y >> 1, side = blockIdx.y & 1, tid = threadIdx.x, NT = blockDim.x;
    const int n_tiles = (Rp >> 2) * 9;
    // a thread owns map rows tr + i*RT and feature rows tq + 9*k (i, k = 0..3): the threads of a quarter-warp then read
    // CONSECUTIVE rows, which the 4-float row padding spreads over all 32 banks (rows 4tr..4tr+3 would sit 528 floats apart:
    // two bank groups, 10 wavefronts per LDS.128 -- measured, profiles/r2_stem_train_ncu.md)
    const int RT = Rp >> 2;
    const int tr = tid / 9, tq = tid - tr * 9;
    const bool worker = tid < n_tiles;
    const int warp = tid >> 5, lane = tid & 31, n_warps = NT >> 5;
    const float* feat = (side == 0 ? x : y) + (size_t)b * kStC * Hf * Wf;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int w0 = 0; w0 < Wf; w0 += kStWC) {
        __syncthreads();
        for (int r = warp; r < Rp + kStQ; r += n_warps) {    // a warp stages whole rows (map rows, then feature rows)
            const float* src = nullptr;
            int shift = 0, lim = 0;
            float* dst;
            if (r < Rp) {
                dst = Ms + (size_t)r * kStWS;
                if (r < R) {
                    const int o = r / 9, kd = (r % 9) / 3, kw = r % 3;
                    const size_t row = (size_t)(b * O + o) * Hf + h;
                    if (side == 0) { src = tmap + (row * 9 + kd * 3 + kw) * Wf; shift = 1 - kw; lim = Wf; }
                    else { src = umap + (row * 6 + kd * 2 + (kw == 2 ? 1 : 0)) * (Wf + 4); shift = kd - kw + 2; lim = Wf + 4; }
                }
            } else {
                const int q = r - Rp, c = q / 3, kh = q - 3 * c, hh = h + kh - 1;
                dst = Fs + (size_t)q * kStWS;
                if (hh >= 0 && hh < Hf) { src = feat + ((size_t)c * Hf + hh) * Wf; lim = Wf; }
            }
#pragma unroll
            for (int k = 0; k < kStWC / 32; ++k) {
                const int j = lane + 32 * k, idx = w0 + j + shift;
                dst[j] = (src != nullptr && idx >= 0 && idx < lim && w0 + j < Wf) ? __ldg(src + idx) : 0.f;
            }
        }
        __syncthreads();
        if (worker) {
            const float* mp = Ms + (size_t)tr * kStWS;
            const float* fp = Fs + (size_t)tq * kStWS;
            for (int j = 0; j < kStWC; j += 4) {
                float4 m[4], f[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    m[i] = *reinterpret_cast<const float4*>(mp + (size_t)i * RT * kStWS + j);
                    f[i] = *reinterpret_cast<const float4*>(fp + (size_t)i * 9 * kStWS + j);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        acc[i][k] = __fmaf_rn(m[i].x, f[k].x, __fmaf_rn(m[i].y, f[k].y, __fmaf_rn(m[i].z, f[k].z, __fmaf_rn(m[i].w, f[k].w, acc[i][k]))));
            }
        }
    }
    if (worker) {
        float* dst = part + ((size_t)(b * Hf + h) * 2 + side) * (size_t)R * kStQ;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = tr + i * RT;
            if (r < R)
#pragma unroll
                for (int k = 0; k < 4; ++k) dst[(size_t)r * kStQ + tq + 9 * k] = acc[i][k];
        }
    }
}

// gW[o, side*C + c, kd, kh, kw] = sum over (b,h) of part[...][side][(o,kd,kw)][(c,kh)], fixed order, fp64: a warp per 32
// consecutive outputs walks the partials (coalesced 128-byte rows), 8 warps of a CTA take every 8th partial and are added
// in a fixed order through shared memory.  grid ceil(2*R*Q / 32), 256 threads.
__global__ void __launch_bounds__(256)
stem_bwd_weight_final_kernel(const float* __restrict__ part, float* __restrict__ gw, int n_bh, int O) {
    const int R = 9 * O, n_out = 2 * R * kStQ;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;                    // output index over [side][r][q]
    __shared__ double red[8][32];
    double a = 0.0;
    if (i < n_out) {
        const int side = i / (R * kStQ), rq = i - side * R * kStQ;
        for (int k = warp; k < n_bh; k += 8) a += (double)part[((size_t)k * 2 + side) * R * kStQ + rq];
    }
    red[warp][lane] = a;
    __syncthreads();
    if (warp == 0 && i < n_out) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][lane];
        const int side = i / (R * kStQ), rq = i - side * R * kStQ;
        const int r = rq / kStQ, q = rq - r * kStQ;
        const int o = r / 9, kd = (r % 9) / 3, kw = r % 3, c = q / 3, kh = q - 3 * c;
        gw[((((size_t)o * 2 * kStC + side * kStC + c) * 3 + kd) * 3 + kh) * 3 + kw] = (float)t;
    }
}

// ---- host -------------------------------------------------------------------------------------------------------------
static int check_stem_train(const char* who, int B, int C, int O, int Df, int Hf, int Wf) {
    if (B <= 0 || O <= 0 || Df <= 0 || Hf <= 0 || Wf <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    if (C != kStC || O > 32 || Df < 3 || Wf < 8 || Wf % 4 != 0 || Wf > 1016 || B > 32767 || O > 65535 || Hf > 65535)
        return fail(RAG_E_SHAPE, "%s: needs C == 12, O <= 32, Df >= 3, 8 <= Wf <= 1016 with Wf %% 4 == 0, B <= 32767, Hf <= 65535 (got B=%d C=%d O=%d Df=%d Hf=%d Wf=%d)",
                    who, B, C, O, Df, Hf, Wf);
    if ((size_t)B * O * Df * Hf * Wf >= ((size_t)1 << 40)) return fail(RAG_E_SHAPE, "%s: tensor too large", who);
    return RAG_OK;
}

size_t cv_stem_bwd_workspace_bytes(int B, int C, int O, int Hf, int Wf) {
    if (C != kStC || B <= 0 || O <= 0 || Hf <= 0 || Wf <= 0) return 0;
    const size_t rows = (size_t)B * O * Hf;
    return (rows * 9 * Wf + rows * 6 * (Wf + 4) + (size_t)B * Hf * 2 * 9 * O * kStQ) * sizeof(float);
}

// gx, gy [B,C,Hf,Wf] (nullable pair), gw [O,2C,3,3,3] (nullable) from g, z [B,O,Df,Hf,Wf], consts [O][7], x, y, w.
int cv_stem_bwd(const float* g, const float* out, const float* consts, const float* x, const float* y, const float* w,
                float* gx, float* gy, float* gw, float* workspace, int B, int C, int O, int Df, int Hf, int Wf, cudaStream_t st) {
    if (!g || !out || !consts || !workspace) return fail(RAG_E_NULL, "cv_stem_bwd: null pointer");
    if ((gx == nullptr) != (gy == nullptr)) return fail(RAG_E_NULL, "cv_stem_bwd: gx and gy go together");
    if (gx && !w) return fail(RAG_E_NULL, "cv_stem_bwd: the input gradients need the weight");
    if (gw && (!x || !y)) return fail(RAG_E_NULL, "cv_stem_bwd: the weight gradient needs x and y");
    if (int e = check_stem_train("cv_stem_bwd", B, C, O, Df, Hf, Wf)) return e;
    if (!aligned(workspace, 16) || (gx && (!aligned(gx, 16) || !aligned(gy, 16))))
        return fail(RAG_E_ALIGN, "cv_stem_bwd: workspace, gx, gy must be 16-byte aligned");
    const size_t rows = (size_t)B * O * Hf;
    float* tmap = workspace;
    float* umap = tmap + rows * 9 * Wf;
    float* part = umap + rows * 6 * (Wf + 4);
    {
        const int nt = ((Wf + 4 + 31) / 32) * 32;
        const int U = Df % 8 == 0 ? 8 : Df % 4 == 0 ? 4 : Df % 2 == 0 ? 2 : 1;   // rows per batch: must divide Df
        const size_t smem = ((size_t)2 * U + 5) * Wf * sizeof(float);
        if (U == 8) stem_bwd_maps_kernel<8><<<dim3(Hf, O, B), nt, smem, st>>>(g, out, consts, tmap, umap, O, Df, Hf, Wf);
        else if (U == 4) stem_bwd_maps_kernel<4><<<dim3(Hf, O, B), nt, smem, st>>>(g, out, consts, tmap, umap, O, Df, Hf, Wf);
        else if (U == 2) stem_bwd_maps_kernel<2><<<dim3(Hf, O, B), nt, smem, st>>>(g, out, consts, tmap, umap, O, Df, Hf, Wf);
        else stem_bwd_maps_kernel<1><<<dim3(Hf, O, B), nt, smem, st>>>(g, out, consts, tmap, umap, O, Df, Hf, Wf);
        if (int e = check_launch("cv_stem_bwd(maps)")) return e;
    }
    const int R = 9 * O, Rp = (R + 3) & ~3;
    if (gx) {
        const size_t smem = (std::max((size_t)R * kStWC, (size_t)kStTH * 12 * 128) + (size_t)3 * R * 16) * sizeof(float);
        cudaError_t e = cudaFuncSetAttribute(stem_bwd_inputs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail((int)e, "cv_stem_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        stem_bwd_inputs_kernel<<<dim3((Wf + kStWC - 1) / kStWC, (Hf + kStTH - 1) / kStTH, 2 * B), 256, smem, st>>>(tmap, umap, w, gx, gy, O, Hf, Wf);
        if (int rc = check_launch("cv_stem_bwd(inputs)")) return rc;
    }
    if (gw) {
        const size_t smem = ((size_t)Rp * kStWS + (size_t)kStQ * kStWS) * sizeof(float);
        cudaError_t e = cudaFuncSetAttribute(stem_bwd_weight_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail((int)e, "cv_stem_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        const int nt = (((Rp >> 2) * 9 + 31) / 32) * 32;
        stem_bwd_weight_kernel<<<dim3(Hf, 2 * B), nt, smem, st>>>(tmap, umap, x, y, part, O, Hf, Wf);
        if (int rc = check_launch("cv_stem_bwd(weight)")) return rc;
        stem_bwd_weight_final_kernel<<<(2 * R * kStQ + 31) / 32, 256, 0, st>>>(part, gw, B * Hf, O);
        if (int rc = check_launch("cv_stem_bwd(weight final)")) return rc;
    }
    return RAG_OK;
}

}  // namespace rag
