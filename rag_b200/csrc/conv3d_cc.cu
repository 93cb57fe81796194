// The Matching Net's interior 3x3x3 layers: ConvBR_3d(C, O, 3, 1, 1) = bias-free Conv3d C -> O, stride 1, zero padding 1,
// then BatchNorm3d + ReLU (src/automl/operations_3d.py:31-47).  In the growable Network this is `stem3d1` (12 -> 12 at the
// volume's resolution) and every `conv_3x3` op of the Cell_3d's (4 / 8 / 16 channels at levels 3 / 6 / 12):
//     z[b,o,p] = sum_{c,k} w[o,c,k] x[b,c,p+k-1]                                   (forward)
//     gx[b,c,p] = sum_{o,k} w[o,c,k] gz[b,o,p-k+1] = sum_{o,k} w[o,c,26-k] gz[b,o,p+k-1]   (data gradient: the forward
//                 stencil on gz with the weights transposed to [C,O] and flipped in k -- the same kernel, FLIP = true)
//     gw[o,c,k] = sum_{b,p} gz[b,o,p] x[b,c,p+k-1]                                   (weight gradient)
// All channel counts are compile-time: (C, O) in {(4,4), (8,8), (12,12)}; anything else is RAG_E_SHAPE.  (16,16), the level-12
// op, was measured slower than cuDNN (TF32) at its shapes -- a grid of 24 CTAs at B=4 288x576 -- and is not compiled.
//
// Forward / data gradient.  A CTA of 128 threads owns an 8 (h) x 64 (w) column of up to 8 output planes of one pair and
// walks them along d; a thread owns 4 adjacent w of one h for ALL O output channels (4*O accumulators).  A unit of work is
// one input channel's three planes d-1, d, d+1 (10 rows x 72 columns each, halo included, zero-filled outside the volume by
// cp.async zfill); units stream through a 3-slot shared-memory ring filled two units ahead, one block barrier per unit.
// The weights sit in shared memory as [c][k][o] (loaded once per CTA): one LDS.128 broadcast gives four output channels'
// weight for one tap, against the thread's six inputs of a row -- 16 FFMA per weight load.  No constant memory (last_conv.cu's
// slots already take 57 KB of it), so these kernels are stateless and capturable.
//
// Weight gradient.  O*C*27 sums.  A thread owns one (c, kd, kh) and its 3 (kw) x O sums; the CTA walks a 2 (h) x 64 (w)
// column of up to 8 planes per tile (x: the three planes around d of all C channels, 4 rows each; gz: plane d of all O
// channels), double-buffered by cp.async.  Every thread walks the same positions, so the gz loads are broadcasts and the
// thread's x row slides along w in registers (one LDS.128 per four positions).  A fixed grid of kCcWgGroups CTAs takes
// tiles blockIdx.x, blockIdx.x + G, ... and writes one fp32 partial per sum; a final kernel adds the partials in a fixed
// order in fp64: bitwise repeatable.
#include <cuda_pipeline.h>

#include <algorithm>

#include "common.cuh"

namespace rag {

constexpr int kCcHT = 8, kCcWT = 64, kCcDT = 8;                // forward tile: 8 h x 64 w x 8 planes
constexpr int kCcRS = 76;                                        // row stride (floats): 18 vectors w0-4 .. w0+67, 16-byte rows;
                                                                 // 76 = 12 mod 32 puts 8 consecutive rows in distinct bank groups
constexpr int kCcUnit = 3 * (kCcHT + 2) * kCcRS;                 // one channel, three planes
constexpr int kCcRing = 3;
constexpr int kCcThreads = 128;
constexpr int kCcWgHT = 2, kCcWgDT = 8;                          // weight-gradient tile: 2 h x 64 w x 8 planes
constexpr int kCcWgGroups = 296;                                 // CTAs (= partials per sum) of the weight gradient

__host__ __device__ constexpr int cc_wg_threads(int C) { return ((C * 9 + 31) / 32) * 32; }
__host__ __device__ constexpr int cc_wg_slot(int C, int O) { return 3 * C * (kCcWgHT + 2) * kCcRS + O * kCcWgHT * kCcWT; }

// grid: x = ceil(W/64), y = ceil(H/8), z = B * ceil(D/8); 128 threads.  smem: kCcRing * kCcUnit + CI*27*CO floats.
// FLIP = false: w [CO][CI][27] (forward).  FLIP = true: w [CI][CO][27] read at tap 26-k (data gradient).
template <int CI, int CO, bool FLIP>
__global__ void __launch_bounds__(kCcThreads, 4)
conv3d_cc_fwd_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ scale,
                     const float* __restrict__ shift, int relu, float* __restrict__ out, int D, int H, int W, int n_dt) {
    static_assert(CO % 4 == 0, "output channels come in groups of four");
    extern __shared__ __align__(16) float cc_smem[];
    float* ring = cc_smem;
    float* wsm = cc_smem + kCcRing * kCcUnit;
    const int tid = threadIdx.x;
    const int b = blockIdx.z / n_dt, dt = blockIdx.z - b * n_dt;
    const int d0 = dt * kCcDT, h0 = blockIdx.y * kCcHT, w0 = blockIdx.x * kCcWT;
    const int nsteps = min(kCcDT, D - d0);
    const size_t plane = (size_t)H * W, chan = (size_t)D * plane;
    const float* inb = in + (size_t)b * CI * chan;

    for (int i = tid; i < CI * 27 * CO; i += kCcThreads) {       // [ci][k][co]
        const int ci = i / (27 * CO), rem = i - ci * 27 * CO, k = rem / CO, co = rem - k * CO;
        wsm[i] = FLIP ? __ldg(w + ((size_t)ci * CO + co) * 27 + 26 - k) : __ldg(w + ((size_t)co * CI + ci) * 27 + k);
    }

    // copy slots of a thread: vector i = tid + 128 s of a unit (540 = 3 planes x 10 rows x 18 vectors); the offset inside the
    // channel relative to (plane d-1, row h0-1, column w0-4) and the smem offset are the same for every unit
    constexpr int kVecs = 3 * (kCcHT + 2) * 18, kSlots = (kVecs + kCcThreads - 1) / kCcThreads;
    int goff[kSlots], soff[kSlots];
    unsigned okhw = 0, kp1 = 0, kp2 = 0;
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
        const int i = tid + kCcThreads * s;
        const int kp = i / ((kCcHT + 2) * 18), rem = i - kp * (kCcHT + 2) * 18, r = rem / 18, v = rem - r * 18;
        const int gh = h0 - 1 + r, gw = w0 - 4 + 4 * v;
        goff[s] = kp * (int)plane + gh * W + gw;                  // 3*H*W < 2^31 (checked on the host)
        soff[s] = (kp * (kCcHT + 2) + r) * kCcRS + 4 * v;
        okhw |= (i < kVecs && gh >= 0 && gh < H && gw >= 0 && gw < W) ? 1u << s : 0u;   // W % 4 == 0
        kp1 |= kp == 1 ? 1u << s : 0u;
        kp2 |= kp == 2 ? 1u << s : 0u;
    }
    const int total = nsteps * CI;
    auto issue = [&](int u) {
        if (u < total) {
            const int st = u / CI, ci = u - st * CI, d = d0 + st;
            const float* src = inb + (size_t)ci * chan + (ptrdiff_t)(d - 1) * (ptrdiff_t)plane;
            float* dst = ring + (u % kCcRing) * kCcUnit;
            const bool p0 = d - 1 >= 0, p2 = d + 1 < D;
#pragma unroll
            for (int s = 0; s < kSlots; ++s) {
                if (tid + kCcThreads * s < kVecs) {
                    const bool ok = (okhw >> s & 1u) && ((kp1 >> s & 1u) || ((kp2 >> s & 1u) ? p2 : p0));
                    __pipeline_memcpy_async(dst + soff[s], ok ? src + goff[s] : inb, 16, ok ? 0 : 16);
                }
            }
        }
        __pipeline_commit();
    };
    issue(0);
    issue(1);

    const int tx = tid & 15, ty = tid >> 4;
    float acc[CO][4];
#pragma unroll
    for (int o = 0; o < CO; ++o)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[o][j] = 0.f;
    const int h = h0 + ty, wo = w0 + 4 * tx;

#pragma unroll 1
    for (int u = 0; u < total; ++u) {
        __pipeline_wait_prior(1);
        __syncthreads();                                          // unit u landed for all threads; all are past unit u-1
        issue(u + 2);                                             // into the slot unit u-1 used
        const int ci = u % CI;
        const float* st = ring + (u % kCcRing) * kCcUnit + ty * kCcRS + 4 * tx;
        const float* ws = wsm + ci * 27 * CO;
#pragma unroll
        for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
                const float* p = st + (kd * (kCcHT + 2) + kh) * kCcRS;
                const float4 m = *reinterpret_cast<const float4*>(p + 4);
                float v[6];
                v[0] = p[3];
                v[1] = m.x; v[2] = m.y; v[3] = m.z; v[4] = m.w;
                v[5] = p[8];
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) {
                    const float* wk = ws + ((kd * 3 + kh) * 3 + kw) * CO;
#pragma unroll
                    for (int g = 0; g < CO / 4; ++g) {
                        const float4 wv = *reinterpret_cast<const float4*>(wk + 4 * g);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            acc[4 * g + 0][j] = __fmaf_rn(wv.x, v[j + kw], acc[4 * g + 0][j]);
                            acc[4 * g + 1][j] = __fmaf_rn(wv.y, v[j + kw], acc[4 * g + 1][j]);
                            acc[4 * g + 2][j] = __fmaf_rn(wv.z, v[j + kw], acc[4 * g + 2][j]);
                            acc[4 * g + 3][j] = __fmaf_rn(wv.w, v[j + kw], acc[4 * g + 3][j]);
                        }
                    }
                }
            }
        }
        if (ci == CI - 1) {                                       // output plane d complete
            const int d = d0 + u / CI;
            if (h < H && wo < W) {
                float* o = out + (((size_t)b * CO * D + d) * H + h) * W + wo;
#pragma unroll
                for (int c = 0; c < CO; ++c) {
                    float4 r = make_float4(acc[c][0], acc[c][1], acc[c][2], acc[c][3]);
                    if (scale) {
                        const float sc = __ldg(scale + c), sh = __ldg(shift + c);
                        r.x = __fmaf_rn(r.x, sc, sh); r.y = __fmaf_rn(r.y, sc, sh); r.z = __fmaf_rn(r.z, sc, sh); r.w = __fmaf_rn(r.w, sc, sh);
                    }
                    if (relu) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
                    *reinterpret_cast<float4*>(o + (size_t)c * chan) = r;
                }
            }
#pragma unroll
            for (int c = 0; c < CO; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[c][j] = 0.f;
        }
    }
}

// Weight-gradient partials: part [G][CO][CI][27].  grid G (<= kCcWgGroups), cc_wg_threads(CI) threads.
// smem: 2 slots of cc_wg_slot(CI, CO) floats = x [3 planes][CI][4 rows][76] | gz [CO][2 rows][64].
template <int CI, int CO>
__global__ void __launch_bounds__(cc_wg_threads(CI), 2)
conv3d_cc_wgrad_kernel(const float* __restrict__ gz, const float* __restrict__ in, float* __restrict__ part,
                       int D, int H, int W, int n_dt, int n_ht, int n_wt, int n_tiles) {
    constexpr int NT = cc_wg_threads(CI), SLOT = cc_wg_slot(CI, CO);
    constexpr int RX = kCcWgHT + 2;
    constexpr int kXV = 3 * CI * RX * 18, kGV = CO * kCcWgHT * 16;   // vectors per step
    extern __shared__ __align__(16) float wg_smem[];
    const int tid = threadIdx.x, G = gridDim.x;
    const size_t plane = (size_t)H * W, chan = (size_t)D * plane;

    // the step stream: tile t = blockIdx.x + G*j, plane d0 + s of it
    int t_issue = blockIdx.x, s_issue = 0, n_issued = 0;
    auto tile_of = [&](int t, int& b, int& d0, int& h0, int& w0, int& ns) {
        int r = t;
        const int wt = r % n_wt; r /= n_wt;
        const int ht = r % n_ht; r /= n_ht;
        const int dt = r % n_dt; b = r / n_dt;
        d0 = dt * kCcWgDT; h0 = ht * kCcWgHT; w0 = wt * kCcWT;
        ns = min(kCcWgDT, D - d0);
    };
    auto issue = [&]() {
        if (t_issue < n_tiles) {
            int b, d0, h0, w0, ns;
            tile_of(t_issue, b, d0, h0, w0, ns);
            const int d = d0 + s_issue;
            float* dst = wg_smem + (n_issued & 1) * SLOT;
            const float* xb = in + (size_t)b * CI * chan;
            const float* gb = gz + (size_t)b * CO * chan;
            for (int i = tid; i < kXV + kGV; i += NT) {
                const float* src;
                float* sd;
                bool ok;
                if (i < kXV) {                                    // [kp][ci][r][v]
                    const int kp = i / (CI * RX * 18), r1 = i - kp * CI * RX * 18, ci = r1 / (RX * 18), r2 = r1 - ci * RX * 18, r = r2 / 18, v = r2 - r * 18;
                    const int gd = d - 1 + kp, gh = h0 - 1 + r, gw = w0 - 4 + 4 * v;
                    ok = gd >= 0 && gd < D && gh >= 0 && gh < H && gw >= 0 && gw < W;
                    src = xb + (size_t)ci * chan + (size_t)(ok ? gd : 0) * plane + (size_t)(ok ? gh * W + gw : 0);
                    sd = dst + ((kp * CI + ci) * RX + r) * kCcRS + 4 * v;
                } else {                                          // [co][r][v]
                    const int j = i - kXV, co = j / (kCcWgHT * 16), r1 = j - co * kCcWgHT * 16, r = r1 / 16, v = r1 - r * 16;
                    const int gh = h0 + r, gw = w0 + 4 * v;
                    ok = gh < H && gw < W;
                    src = gb + (size_t)co * chan + (size_t)d * plane + (size_t)(ok ? gh * W + gw : 0);
                    sd = dst + 3 * CI * RX * kCcRS + (co * kCcWgHT + r) * kCcWT + 4 * v;
                }
                __pipeline_memcpy_async(sd, src, 16, ok ? 0 : 16);
            }
            if (++s_issue == ns) { s_issue = 0; t_issue += G; }
        }
        ++n_issued;
        __pipeline_commit();
    };

    const bool worker = tid < CI * 9;
    const int c = worker ? tid / 9 : 0, kd = worker ? (tid % 9) / 3 : 0, kh = worker ? tid % 3 : 0;
    float acc[3][CO];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int o = 0; o < CO; ++o) acc[k][o] = 0.f;

    int n_steps = 0;
    for (int t = blockIdx.x; t < n_tiles; t += G) {
        int b, d0, h0, w0, ns;
        tile_of(t, b, d0, h0, w0, ns);
        n_steps += ns;
    }
    issue();
#pragma unroll 1
    for (int step = 0; step < n_steps; ++step) {
        issue();                                                  // next step into the other slot (freed by the barrier below)
        __pipeline_wait_prior(1);
        __syncthreads();
        if (worker) {
            const float* xs = wg_smem + (step & 1) * SLOT + ((kd * CI + c) * RX + kh) * kCcRS;
            const float* gs = wg_smem + (step & 1) * SLOT + 3 * CI * RX * kCcRS;
#pragma unroll
            for (int r = 0; r < kCcWgHT; ++r) {
                const float* xr = xs + r * kCcRS;
                float4 prev = *reinterpret_cast<const float4*>(xr);
                float4 cur = *reinterpret_cast<const float4*>(xr + 4);
#pragma unroll 2
                for (int v = 0; v < 16; ++v) {
                    const float4 nxt = *reinterpret_cast<const float4*>(xr + 4 * v + 8);
                    const float x0 = prev.w, x1 = cur.x, x2 = cur.y, x3 = cur.z, x4 = cur.w, x5 = nxt.x;
#pragma unroll
                    for (int o = 0; o < CO; ++o) {
                        const float4 gv = *reinterpret_cast<const float4*>(gs + (o * kCcWgHT + r) * kCcWT + 4 * v);
                        acc[0][o] = __fmaf_rn(gv.w, x3, __fmaf_rn(gv.z, x2, __fmaf_rn(gv.y, x1, __fmaf_rn(gv.x, x0, acc[0][o]))));
                        acc[1][o] = __fmaf_rn(gv.w, x4, __fmaf_rn(gv.z, x3, __fmaf_rn(gv.y, x2, __fmaf_rn(gv.x, x1, acc[1][o]))));
                        acc[2][o] = __fmaf_rn(gv.w, x5, __fmaf_rn(gv.z, x4, __fmaf_rn(gv.y, x3, __fmaf_rn(gv.x, x2, acc[2][o]))));
                    }
                    prev = cur;
                    cur = nxt;
                }
            }
        }
        __syncthreads();                                          // the slot is free for the issue two steps on
    }
    if (worker) {
        float* pp = part + (size_t)blockIdx.x * CO * CI * 27;
#pragma unroll
        for (int o = 0; o < CO; ++o)
#pragma unroll
            for (int k = 0; k < 3; ++k) pp[((o * CI + c) * 3 + kd) * 9 + kh * 3 + k] = acc[k][o];
    }
}

// gw[i] = sum_g part[g][i], g ascending, fp64
__global__ void __launch_bounds__(256) conv3d_cc_wgrad_final_kernel(const float* __restrict__ part, float* __restrict__ gw, int n, int G) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double a = 0.0;
    for (int g = 0; g < G; ++g) a += (double)part[(size_t)g * n + i];
    gw[i] = (float)a;
}

// ---- host ---------------------------------------------------------------------------------------------------------------
static bool cc_pair(int C, int O) { return C == O && (C == 4 || C == 8 || C == 12); }

static int cc_check(const char* who, int B, int C, int O, int D, int H, int W) {
    if (B <= 0 || C <= 0 || O <= 0 || D <= 0 || H <= 0 || W <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    if (!cc_pair(C, O)) return fail(RAG_E_SHAPE, "%s: (C, O) = (%d, %d) is not compiled; have (4,4), (8,8), (12,12)", who, C, O);
    if (W % 4 != 0) return fail(RAG_E_SHAPE, "%s: W=%d must be a multiple of 4", who, W);
    if (3LL * H * W + 68 >= (1LL << 31)) return fail(RAG_E_SHAPE, "%s: 3*H*W must be < 2^31", who);
    if ((long long)B * ((D + kCcDT - 1) / kCcDT) > 65535 || (H + kCcWgHT - 1) / kCcWgHT > 65535)
        return fail(RAG_E_SHAPE, "%s: B*ceil(D/8) and ceil(H/2) must be <= 65535", who);
    if ((long long)B * ((D + kCcWgDT - 1) / kCcWgDT) * ((H + kCcWgHT - 1) / kCcWgHT) * ((W + kCcWT - 1) / kCcWT) >= (1LL << 31))
        return fail(RAG_E_SHAPE, "%s: too many weight-gradient tiles", who);
    return RAG_OK;
}

template <int CI, int CO, bool FLIP>
static int cc_launch_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                         int B, int D, int H, int W, cudaStream_t st) {
    auto k = conv3d_cc_fwd_kernel<CI, CO, FLIP>;
    const size_t smem = ((size_t)kCcRing * kCcUnit + (size_t)CI * 27 * CO) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d_cc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int n_dt = (D + kCcDT - 1) / kCcDT;
    k<<<dim3((W + kCcWT - 1) / kCcWT, (H + kCcHT - 1) / kCcHT, B * n_dt), kCcThreads, smem, st>>>(in, w, scale, shift, relu, out, D, H, W, n_dt);
    return check_launch(FLIP ? "conv3d_cc_bwd(data)" : "conv3d_cc_fwd");
}

template <int CI, int CO>
static int cc_launch_wgrad(const float* gz, const float* in, float* gw, float* part, int B, int D, int H, int W, cudaStream_t st) {
    const int n_dt = (D + kCcWgDT - 1) / kCcWgDT, n_ht = (H + kCcWgHT - 1) / kCcWgHT, n_wt = (W + kCcWT - 1) / kCcWT;
    const int n_tiles = B * n_dt * n_ht * n_wt;
    const int G = std::min(kCcWgGroups, n_tiles);                 // a function of the shape only: repeatable on any device
    auto k = conv3d_cc_wgrad_kernel<CI, CO>;
    const size_t smem = 2 * (size_t)cc_wg_slot(CI, CO) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d_cc_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    k<<<G, cc_wg_threads(CI), smem, st>>>(gz, in, part, D, H, W, n_dt, n_ht, n_wt, n_tiles);
    if (int rc = check_launch("conv3d_cc_bwd(weight)")) return rc;
    const int n = CO * CI * 27;
    conv3d_cc_wgrad_final_kernel<<<(n + 255) / 256, 256, 0, st>>>(part, gw, n, G);
    return check_launch("conv3d_cc_bwd(weight final)");
}

int conv3d_cc_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                  int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!in || !w || !out || (scale == nullptr) != (shift == nullptr)) return fail(RAG_E_NULL, "conv3d_cc_fwd: null pointer (scale and shift go together)");
    if (int rc = cc_check("conv3d_cc_fwd", B, C, O, D, H, W)) return rc;
    if (!aligned(in, 16) || !aligned(out, 16) || !aligned(w, 4)) return fail(RAG_E_ALIGN, "conv3d_cc_fwd: in/out must be 16-byte aligned");
    switch (C) {
        case 4: return cc_launch_fwd<4, 4, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
        case 8: return cc_launch_fwd<8, 8, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
        default: return cc_launch_fwd<12, 12, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
    }
}

size_t conv3d_cc_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W) {
    if (!cc_pair(C, O) || B <= 0 || D <= 0 || H <= 0 || W <= 0) return 0;
    return (size_t)kCcWgGroups * O * C * 27 * sizeof(float);
}

int conv3d_cc_bwd(const float* gz, const float* in, const float* w, float* gin, float* gw, float* workspace,
                  int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!gz || (gin && !w) || (gw && (!in || !workspace))) return fail(RAG_E_NULL, "conv3d_cc_bwd: null pointer");
    if (int rc = cc_check("conv3d_cc_bwd", B, C, O, D, H, W)) return rc;
    if (!aligned(gz, 16) || (in && !aligned(in, 16)) || (gin && !aligned(gin, 16)) || (w && !aligned(w, 4)) || (workspace && !aligned(workspace, 4)))
        return fail(RAG_E_ALIGN, "conv3d_cc_bwd: gz/in/gin must be 16-byte aligned");
    if (gin) {
        int rc;
        switch (C) {
            case 4: rc = cc_launch_fwd<4, 4, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st); break;
            case 8: rc = cc_launch_fwd<8, 8, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st); break;
            default: rc = cc_launch_fwd<12, 12, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st); break;
        }
        if (rc) return rc;
    }
    if (gw) {
        switch (C) {
            case 4: return cc_launch_wgrad<4, 4>(gz, in, gw, workspace, B, D, H, W, st);
            case 8: return cc_launch_wgrad<8, 8>(gz, in, gw, workspace, B, D, H, W, st);
            default: return cc_launch_wgrad<12, 12>(gz, in, gw, workspace, B, D, H, W, st);
        }
    }
    return RAG_OK;
}

}  // namespace rag
