// Training-mode BatchNorm3d + ReLU on a convolution output z [B,O,D,H,W], for the fused stem (cv_stem_train.cu) and the
// interior ConvBR_3d layers (conv3d_cc.cu).  Forward: moments of z -> bn [O][4] = (scale, shift, mean, rstd), running
// estimates -> out = max(fma(z, scale, shift), 0).  Backward, with g' = g [fma(z, scale, shift) > 0] (the forward's own ReLU
// decision, bit for bit) and zh = (z - mean) * rstd: (sum g', sum g' zh) -> a = gamma*rstd, m1 = mean(g'), m2 = mean(g' zh)
// (m1 = m2 = 0 in eval) -> gz = a (g' - m1 - zh m2).  In train mode the -a (m1 + zh m2) term reaches every element, also
// where the ReLU is off, so the backward needs z, not only the output.  Fixed-order reductions: bitwise repeatable.
#include <algorithm>

#include "bn3d.cuh"
#include "common.cuh"

namespace rag {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// rows[B,H,O,2] fp64 = per (b,o,h) row (sum z, sum z^2).  grid (H, O, B), 256 threads; W % 4 == 0.
// The fp32 part (four elements at a time) works on z - k, k = the row's first element: var = E[z^2] - mean^2 cancels all but
// a std^2/mean^2 share of the fp32 partials of z^2 itself, so their rounding would reach the variance magnified (mean/std)^2
// times.  The row's raw sums are restored in fp64, where that cancellation is harmless.
__global__ void __launch_bounds__(256)
bn3d_moments_rows_kernel(const float* __restrict__ z, double* __restrict__ rows, int O, int D, int H, int W) {
    const int h = blockIdx.x, o = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const int Wv = W >> 2;
    const size_t plane = (size_t)H * W;
    const size_t base = ((size_t)(b * O + o) * D) * plane + (size_t)h * W;
    const float k = __ldg(z + base);
    double s0 = 0.0, s1 = 0.0;
    for (int i = tid; i < D * Wv; i += 256) {
        const int d = i / Wv, v = i - d * Wv;
        float4 zv = __ldg(reinterpret_cast<const float4*>(z + base + (size_t)d * plane + 4 * v));   // just written: L2
        zv.x -= k; zv.y -= k; zv.z -= k; zv.w -= k;
        const float a = (zv.x + zv.y) + (zv.z + zv.w);
        const float q = __fmaf_rn(zv.x, zv.x, zv.y * zv.y) + __fmaf_rn(zv.z, zv.z, zv.w * zv.w);
        s0 += (double)a;
        s1 += (double)q;
    }
    __shared__ double red[2][8];
    s0 = warp_sum(s0); s1 = warp_sum(s1);
    if ((tid & 31) == 0) { red[0][tid >> 5] = s0; red[1][tid >> 5] = s1; }
    __syncthreads();
    if (tid == 0) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { a0 += red[0][i]; a1 += red[1][i]; }
        const double kd = (double)k, m = (double)D * W;       // sum z = a0 + m k, sum z^2 = a1 + 2 k a0 + m k^2
        double* r = rows + ((size_t)(b * H + h) * O + o) * 2;
        r[0] = a0 + m * kd; r[1] = a1 + kd * (2.0 * a0 + m * kd);
    }
}

// z <- max(fma(z, scale[o], shift[o]), 0) in place, scale / shift = columns 0 / 1 of bn [O][4].  grid-stride over float4;
// n4 = B*O*D*H*W / 4, chan4 = D*H*W / 4
__global__ void __launch_bounds__(256)
bn3d_relu_kernel(float* __restrict__ z, const float* __restrict__ bn, size_t n4, size_t chan4, int O) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (size_t)gridDim.x * 256) {
        const int o = (int)((i / chan4) % O);
        const float sc = __ldg(bn + 4 * o), sh = __ldg(bn + 4 * o + 1);
        float4 v = reinterpret_cast<float4*>(z)[i];
        v.x = fmaxf(__fmaf_rn(v.x, sc, sh), 0.f); v.y = fmaxf(__fmaf_rn(v.y, sc, sh), 0.f);
        v.z = fmaxf(__fmaf_rn(v.z, sc, sh), 0.f); v.w = fmaxf(__fmaf_rn(v.w, sc, sh), 0.f);
        reinterpret_cast<float4*>(z)[i] = v;
    }
}

// Per-channel finaliser (one tiny launch instead of ~15 elementwise torch kernels): sums [O][2] fp64 = (sum z, sum z^2) when
// batch != 0 -> bn [O][4].  With batch and update the running estimates move as nn.BatchNorm's do in train(): r = (1-f) r +
// f * batch value, variance unbiased (n/(n-1)).
__global__ void bn3d_finalize_kernel(const double* __restrict__ sums, const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ running_mean, float* __restrict__ running_var, float* __restrict__ bn,
                                     int O, double n, double eps, double f, int batch, int update) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O) return;
    double mean, var;
    if (batch) {
        mean = sums[2 * o] / n;
        var = fmax(sums[2 * o + 1] / n - mean * mean, 0.0);
        if (update) {
            running_mean[o] = (float)((1.0 - f) * (double)running_mean[o] + f * mean);
            running_var[o] = (float)((1.0 - f) * (double)running_var[o] + f * var * (n / fmax(n - 1.0, 1.0)));
        }
    } else {
        mean = (double)running_mean[o];
        var = (double)running_var[o];
    }
    const float rstd = (float)(1.0 / sqrt(var + eps));
    const float mu = (float)mean;
    const float sc = gamma[o] * rstd;
    bn[4 * o] = sc; bn[4 * o + 1] = beta[o] - mu * sc; bn[4 * o + 2] = mu; bn[4 * o + 3] = rstd;
}

// sums [O][2] fp64 = (sum g', sum g' zh) -> consts [O][7] = (a, m1, m2, scale, shift, mean, rstd), gparam [2][O] = (ggamma, gbeta)
__global__ void bn3d_bwd_consts_kernel(const double* __restrict__ sums, const float* __restrict__ bn, float* __restrict__ consts,
                                       float* __restrict__ gparam, int O, double n, int batch) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O) return;
    const double s0 = sums[2 * o], s1 = sums[2 * o + 1];
    float* c = consts + 7 * o;
    c[0] = bn[4 * o];                                       // a = gamma * rstd = scale
    c[1] = batch ? (float)(s0 / n) : 0.f;
    c[2] = batch ? (float)(s1 / n) : 0.f;
    c[3] = bn[4 * o]; c[4] = bn[4 * o + 1]; c[5] = bn[4 * o + 2]; c[6] = bn[4 * o + 3];
    gparam[o] = (float)s1;                                   // d/d gamma
    gparam[O + o] = (float)s0;                               // d/d beta
}

// per (b,o,h) row  (sum g', sum g'*zh)  ->  rows[B,H,O,2] fp64.  bn [O][4] = (scale, shift, mean, rstd).
// grid (H, O, B), 256 threads; W % 4 == 0.
__global__ void __launch_bounds__(256)
bn3d_bwd_rows_kernel(const float* __restrict__ g, const float* __restrict__ z, const float* __restrict__ bn,
                     double* __restrict__ rows, int O, int D, int H, int W) {
    const int h = blockIdx.x, o = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const int Wv = W >> 2;
    const size_t plane = (size_t)H * W;
    const size_t base = ((size_t)(b * O + o) * D) * plane + (size_t)h * W;
    const float sc = __ldg(bn + 4 * o), sh = __ldg(bn + 4 * o + 1), mu = __ldg(bn + 4 * o + 2), rs = __ldg(bn + 4 * o + 3);
    float s0 = 0.f, s1 = 0.f;
    for (int i = tid; i < D * Wv; i += 256) {
        const int d = i / Wv, v = i - d * Wv;
        const size_t idx = base + (size_t)d * plane + 4 * v;
        const float4 zv = ld_stream(reinterpret_cast<const float4*>(z + idx));
        const float4 gv = ld_stream(reinterpret_cast<const float4*>(g + idx));
        const float g0 = __fmaf_rn(zv.x, sc, sh) > 0.f ? gv.x : 0.f, g1 = __fmaf_rn(zv.y, sc, sh) > 0.f ? gv.y : 0.f;
        const float g2 = __fmaf_rn(zv.z, sc, sh) > 0.f ? gv.z : 0.f, g3 = __fmaf_rn(zv.w, sc, sh) > 0.f ? gv.w : 0.f;
        s0 += (g0 + g1) + (g2 + g3);
        s1 += (g0 * ((zv.x - mu) * rs) + g1 * ((zv.y - mu) * rs)) + (g2 * ((zv.z - mu) * rs) + g3 * ((zv.w - mu) * rs));
    }
    __shared__ double red[2][8];
    double d0 = warp_sum((double)s0), d1 = warp_sum((double)s1);
    if ((tid & 31) == 0) { red[0][tid >> 5] = d0; red[1][tid >> 5] = d1; }
    __syncthreads();
    if (tid == 0) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { a0 += red[0][i]; a1 += red[1][i]; }
        double* r = rows + ((size_t)(b * H + h) * O + o) * 2;
        r[0] = a0; r[1] = a1;
    }
}

// rows[B*H][O][2] -> sums[O][2], fixed order (deterministic).  grid O, 32 threads.
__global__ void bn3d_rows_final_kernel(const double* __restrict__ rows, double* __restrict__ sums, int n_rows, int O) {
    const int o = blockIdx.x, lane = threadIdx.x;
    double a0 = 0.0, a1 = 0.0;
    for (int i = lane; i < n_rows; i += 32) {
        a0 += rows[((size_t)i * O + o) * 2];
        a1 += rows[((size_t)i * O + o) * 2 + 1];
    }
    a0 = warp_sum(a0); a1 = warp_sum(a1);
    if (lane == 0) { sums[2 * o] = a0; sums[2 * o + 1] = a1; }
}

// gz = a (g' - m1 - zh m2) with consts [O][7] = (a, m1, m2, scale, shift, mean, rstd) (bn3d.cuh).  Grid-stride over float4.
__global__ void __launch_bounds__(256)
bn3d_bwd_gz_kernel(const float* __restrict__ g, const float* __restrict__ z, const float* __restrict__ consts, float* __restrict__ gz,
                   size_t n4, size_t chan4, int O) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (size_t)gridDim.x * 256) {
        const int o = (int)((i / chan4) % O);
        const float* cs = consts + 7 * o;
        const float a = __ldg(cs), m1 = __ldg(cs + 1), m2 = __ldg(cs + 2), sc = __ldg(cs + 3), sh = __ldg(cs + 4), mu = __ldg(cs + 5), rs = __ldg(cs + 6);
        const float4 zv = ld_stream(reinterpret_cast<const float4*>(z) + i);
        const float4 gv = ld_stream(reinterpret_cast<const float4*>(g) + i);
        float4 r;
        r.x = bn3d_gz(gv.x, zv.x, a, m1, m2, sc, sh, mu, rs);
        r.y = bn3d_gz(gv.y, zv.y, a, m1, m2, sc, sh, mu, rs);
        r.z = bn3d_gz(gv.z, zv.z, a, m1, m2, sc, sh, mu, rs);
        r.w = bn3d_gz(gv.w, zv.w, a, m1, m2, sc, sh, mu, rs);
        reinterpret_cast<float4*>(gz)[i] = r;
    }
}

// ---- host -------------------------------------------------------------------------------------------------------------
// The fused stem's limits (cv_stem_train.cu), which the routing of both callers is built on
static int check_bn3d(const char* who, int B, int O, int D, int H, int W) {
    if (B <= 0 || O <= 0 || D <= 0 || H <= 0 || W <= 0) return fail(RAG_E_SHAPE, "%s: non-positive dimension", who);
    if (O > 32 || D < 3 || W < 8 || W % 4 != 0 || W > 1016 || B > 32767 || H > 65535)
        return fail(RAG_E_SHAPE, "%s: needs O <= 32, D >= 3, 8 <= W <= 1016 with W %% 4 == 0, B <= 32767, H <= 65535 (got B=%d O=%d D=%d H=%d W=%d)",
                    who, B, O, D, H, W);
    if ((size_t)B * O * D * H * W >= ((size_t)1 << 40)) return fail(RAG_E_SHAPE, "%s: tensor too large", who);
    return RAG_OK;
}

// sums[O][2] (fp64) = (sum z, sum z^2) over (B, D, H, W); rows_ws: fp64 workspace of B*H*O*2 doubles
int bn3d_moments(const float* z, double* sums, double* rows_ws, int B, int O, int D, int H, int W, cudaStream_t st) {
    if (!z || !sums || !rows_ws) return fail(RAG_E_NULL, "bn3d_moments: null pointer");
    if (int e = check_bn3d("bn3d_moments", B, O, D, H, W)) return e;
    if (!aligned(z, 16) || !aligned(sums, 8) || !aligned(rows_ws, 8)) return fail(RAG_E_ALIGN, "bn3d_moments: z must be 16-byte aligned");
    bn3d_moments_rows_kernel<<<dim3(H, O, B), 256, 0, st>>>(z, rows_ws, O, D, H, W);
    if (int e = check_launch("bn3d_moments(rows)")) return e;
    bn3d_rows_final_kernel<<<O, 32, 0, st>>>(rows_ws, sums, B * H, O);
    return check_launch("bn3d_moments(final)");
}

// bn [O][4] from the batch moments (batch != 0) or the running statistics; see bn3d_finalize_kernel
int bn3d_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                  float* bn, int O, double n, double eps, double momentum, int batch, int update, cudaStream_t st) {
    if (!gamma || !beta || !bn || (batch && !sums) || ((!batch || update) && (!running_mean || !running_var)))
        return fail(RAG_E_NULL, "bn3d_finalize: null pointer");
    if (O <= 0 || n < 1.0) return fail(RAG_E_SHAPE, "bn3d_finalize: bad O or n");
    bn3d_finalize_kernel<<<(O + 63) / 64, 64, 0, st>>>(sums, gamma, beta, running_mean, running_var, bn, O, n, eps, momentum, batch, update);
    return check_launch("bn3d_finalize");
}

// z <- relu(z * scale[o] + shift[o]) in place (one fused multiply-add per element: the expression the backward re-evaluates)
int bn3d_relu(float* z, const float* bn, int B, int O, int D, int H, int W, cudaStream_t st) {
    if (!z || !bn) return fail(RAG_E_NULL, "bn3d_relu: null pointer");
    if (int e = check_bn3d("bn3d_relu", B, O, D, H, W)) return e;
    if (!aligned(z, 16)) return fail(RAG_E_ALIGN, "bn3d_relu: z must be 16-byte aligned");
    const size_t chan4 = (size_t)D * H * W / 4, n4 = chan4 * O * B;
    const unsigned grid = (unsigned)std::min<size_t>((n4 + 255) / 256, (size_t)num_sms() * 32);
    bn3d_relu_kernel<<<grid, 256, 0, st>>>(z, bn, n4, chan4, O);
    return check_launch("bn3d_relu");
}

// sums[O][2] (fp64) = (sum g', sum g'*zh) over (B, D, H, W); rows_ws: B*H*O*2 doubles
int bn3d_bwd_sums(const float* g, const float* z, const float* bn, double* sums, double* rows_ws,
                  int B, int O, int D, int H, int W, cudaStream_t st) {
    if (!g || !z || !bn || !sums || !rows_ws) return fail(RAG_E_NULL, "bn3d_bwd_sums: null pointer");
    if (int e = check_bn3d("bn3d_bwd_sums", B, O, D, H, W)) return e;
    if (!aligned(g, 16) || !aligned(z, 16) || !aligned(sums, 8) || !aligned(rows_ws, 8)) return fail(RAG_E_ALIGN, "bn3d_bwd_sums: g/z must be 16-byte aligned");
    bn3d_bwd_rows_kernel<<<dim3(H, O, B), 256, 0, st>>>(g, z, bn, rows_ws, O, D, H, W);
    if (int e = check_launch("bn3d_bwd_sums(rows)")) return e;
    bn3d_rows_final_kernel<<<O, 32, 0, st>>>(rows_ws, sums, B * H, O);
    return check_launch("bn3d_bwd_sums(final)");
}

int bn3d_bwd_consts(const double* sums, const float* bn, float* consts, float* gparam, int O, double n, int batch, cudaStream_t st) {
    if (!sums || !bn || !consts || !gparam) return fail(RAG_E_NULL, "bn3d_bwd_consts: null pointer");
    if (O <= 0 || n < 1.0) return fail(RAG_E_SHAPE, "bn3d_bwd_consts: bad O or n");
    bn3d_bwd_consts_kernel<<<(O + 63) / 64, 64, 0, st>>>(sums, bn, consts, gparam, O, n, batch);
    return check_launch("bn3d_bwd_consts");
}

int bn3d_bwd_gz(const float* g, const float* z, const float* consts, float* gz, int B, int O, int D, int H, int W, cudaStream_t st) {
    if (!g || !z || !consts || !gz) return fail(RAG_E_NULL, "bn3d_bwd_gz: null pointer");
    if (int e = check_bn3d("bn3d_bwd_gz", B, O, D, H, W)) return e;
    if (!aligned(g, 16) || !aligned(z, 16) || !aligned(gz, 16) || !aligned(consts, 4)) return fail(RAG_E_ALIGN, "bn3d_bwd_gz: g/z/gz must be 16-byte aligned");
    const size_t chan4 = (size_t)D * H * W / 4, n4 = chan4 * O * B;
    const unsigned grid = (unsigned)std::min<size_t>((n4 + 255) / 256, (size_t)num_sms() * 16);
    bn3d_bwd_gz_kernel<<<grid, 256, 0, st>>>(g, z, consts, gz, n4, chan4, O);
    return check_launch("bn3d_bwd_gz");
}

}  // namespace rag
