// The interior 3x3x3 ConvBR_3d layers of conv3d_cc.cu on the tensor cores: an implicit GEMM on tcgen05.mma kind::tf32 with
// the fp32 accumulator in tensor memory.  Same (C, O) pairs, same contract, same shape limits (cc_check) as the fp32 kernels.
//     D[m, n] = sum_k A[m, k] B[k, n]:  m = output voxel, n = output channel (O padded to 16 with zero weights),
//     k = (kd, kh, kw, c).  The data gradient is the same kernel with FLIP = true (weights [O][C] flipped in k), as in
//     conv3d_cc_fwd_kernel.
//
// Numerics.  Both operands are rounded to TF32 (10-bit mantissa) with round-to-nearest, ties away (cvt.rna.tf32.f32) as
// they are staged into shared memory; the MMA would otherwise drop the low 13 bits (truncation), which biases every
// product toward zero.  Products are summed in fp32 inside the tensor core, in an order fixed by the hardware and the tap
// order below: bitwise repeatable.  No atomics, no constant memory: stateless and capturable.
//
// Layout.  A CTA owns an Ht x Wt output patch of one batch item and walks up to 8 planes along d.  An input plane of the
// patch (halo included, Wq = Wt + 2 columns per row) sits in shared memory as [c / 4][row * Wq + col][c % 4]: each position
// holds four channels in 16 bytes.  That is the K-major, no-swizzle canonical layout of tcgen05 with one position per
// M row (8 rows of 16 bytes = one core matrix, SBO = 128 bytes), and output position q = row * Wq + col reads tap
// (kh, kw) at q + kh * Wq + kw.  So every tap is a descriptor offset by whole 16-byte positions: the kw = +-1 taps need no
// shifted copies.  The columns q of the two 128-row M tiles that fall on the halo (col >= Wt) are computed and dropped.
// One MMA has K = 8 = two 4-channel k-groups, the second at LBO bytes past the first; the 9 * C / 4 k-groups of a plane,
// ordered (c / 4, kh, kw), are taken in pairs (offsets increase along that order, so LBO > 0).  An odd count leaves one
// k-group alone: its partner is itself (LBO = 0) against zero weights, so the padding reads only values the output already
// depends on.  MMAs per output plane and M tile: 15 / 27 / 42 for C = 4 / 8 / 12.
//
// Pipeline.  Input planes go through a 4-slot ring (planes d-1, d, d+1 in use, d+2 being staged).  Per output plane one
// thread issues the 2 x 3 x NP MMAs and commits them to an mbarrier; meanwhile all threads stage the next plane (LDG,
// rounding, STS.128).  Then the 128 threads read the accumulator (thread t = TMEM lane t = M row t, tcgen05.ld 32x32b),
// apply max?(fma(z, scale, shift), 0) and store.  TMEM: 32 columns (2 tiles x 16) per CTA.
#include <algorithm>
#include <climits>

#include "common.cuh"

namespace rag {

int cc_check(const char* who, int B, int C, int O, int D, int H, int W);   // conv3d_cc.cu

constexpr int kTfThreads = 128;
constexpr int kTfRows = 256;                 // M rows (output positions) per plane: two 128-row MMA tiles
constexpr int kTfMaxWq = 64;                 // widest staged row (Wt <= 62)
constexpr int kTfSlab = 392;                 // positions per (4-channel group, plane) slot: >= kTfRows + 2 * kTfMaxWq + 3
constexpr int kTfRing = 4;
constexpr int kTfDT = 8;                     // planes per CTA (kCcDT: the grid limit of cc_check)
constexpr int kTfN = 16;                     // MMA N: O padded
constexpr int kTfTmemCols = 32;

__host__ __device__ constexpr int tf_np(int CI) { return (9 * (CI / 4) + 1) / 2; }           // MMAs per plane and tile
__host__ __device__ constexpr size_t tf_smem(int CI) {
    return (size_t)kTfRing * (CI / 4) * kTfSlab * 16 + (size_t)3 * tf_np(CI) * 512;
}

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// shared-memory matrix descriptor: no swizzle, K-major (start, LBO, SBO in bytes; bits 46-47 = 1 on sm_100)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// instruction descriptor, kind::tf32: D fp32 (bits 4-5 = 1), A and B tf32 (bits 7-9, 10-12 = 2), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t kTfIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kTfN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__device__ __forceinline__ void mma_tf32(uint32_t dtmem, uint64_t a, uint64_t b, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(dtmem), "l"(a), "l"(b), "r"(kTfIdesc), "r"(accumulate));
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.b32 %0, 1, 0, P;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// grid: x = n_wt, y = n_ht, z = B * ceil(D/8); 128 threads; smem tf_smem(CI).
// FLIP = false: w [CO][CI][27] (forward).  FLIP = true: w [CI][CO][27] read at tap 26-k (data gradient).
template <int CI, int CO, bool FLIP>
__global__ void __launch_bounds__(kTfThreads)
conv3d_cc_tf32_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ scale,
                      const float* __restrict__ shift, int relu, float* __restrict__ out, int D, int H, int W,
                      int Wt, int Ht, int n_dt) {
    static_assert(CI % 4 == 0 && CO <= kTfN, "4-channel k-groups; O fits N = 16");
    constexpr int CG = CI / 4, NP = tf_np(CI), SLOT = CG * kTfSlab * 16;   // bytes of one plane slot
    extern __shared__ __align__(128) unsigned char tf_smem_buf[];
    __shared__ __align__(8) uint64_t mbar;
    __shared__ uint32_t tmem_base;
    float4* ring = reinterpret_cast<float4*>(tf_smem_buf);
    float* bsm = reinterpret_cast<float*>(tf_smem_buf + kTfRing * SLOT);   // [kd][pair][k-group j][n][4]

    const int tid = threadIdx.x, warp = tid >> 5;
    const int b = blockIdx.z / n_dt, d0 = (blockIdx.z - b * n_dt) * kTfDT;
    const int h0 = blockIdx.y * Ht, w0 = blockIdx.x * Wt, Wq = Wt + 2;
    const int ns = min(kTfDT, D - d0);
    const size_t plane = (size_t)H * W, chan = (size_t)D * plane;
    const float* inb = in + (size_t)b * CI * chan;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_addr(&tmem_base)), "r"(kTfTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(&mbar)), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // weights: B for (kd, pair p) = k-groups 2p, 2p+1 of the plane order (c/4, kh, kw); row n, 4 channels per k-group
    for (int i = tid; i < 3 * NP * 2 * kTfN * 4; i += kTfThreads) {
        const int e = i & 3, n = (i >> 2) % kTfN, j = (i / (4 * kTfN)) & 1, pk = i / (8 * kTfN), kd = pk / NP, p = pk - kd * NP;
        const int g = 2 * p + j, cg = g / 9, t = g - 9 * cg, ci = 4 * cg + e, k = kd * 9 + t;
        float v = 0.f;
        if (g < 9 * CG && n < CO)
            v = FLIP ? __ldg(w + ((size_t)ci * CO + n) * 27 + 26 - k) : __ldg(w + ((size_t)n * CI + ci) * 27 + k);
        bsm[i] = tf32_rna(v);
    }

    // stage input plane gd (zeros outside the volume) into the ring slot of relative plane r
    auto stage = [&](int gd, int r) {
        float4* dst = ring + (size_t)(r & (kTfRing - 1)) * (SLOT / 16);
        const bool pd = gd >= 0 && gd < D;
        for (int i = tid; i < CG * kTfSlab; i += kTfThreads) {
            const int cg = i / kTfSlab, pos = i - cg * kTfSlab, row = pos / Wq, col = pos - row * Wq;
            const int gh = h0 - 1 + row, gw = w0 - 1 + col;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pd && row < Ht + 2 && gh >= 0 && gh < H && gw >= 0 && gw < W) {
                const float* s = inb + (size_t)(4 * cg) * chan + (size_t)gd * plane + (size_t)gh * W + gw;
                v.x = tf32_rna(__ldg(s)); v.y = tf32_rna(__ldg(s + chan)); v.z = tf32_rna(__ldg(s + 2 * chan)); v.w = tf32_rna(__ldg(s + 3 * chan));
            }
            dst[i] = v;
        }
    };
    stage(d0 - 1, 0);
    stage(d0, 1);
    stage(d0 + 1, 2);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tmem_base, bar = smem_addr(&mbar), ring_a = smem_addr(ring), b_a = smem_addr(bsm);

    float sc[CO], sh[CO];
#pragma unroll
    for (int o = 0; o < CO; ++o) {
        sc[o] = scale ? __ldg(scale + o) : 1.f;
        sh[o] = scale ? __ldg(shift + o) : 0.f;
    }

#pragma unroll 1
    for (int s = 0; s < ns; ++s) {
        if (tid == 0) {
            fence_after_sync();
#pragma unroll 1
            for (int mt = 0; mt < kTfRows / 128; ++mt) {
                uint32_t acc = 0;
#pragma unroll 1
                for (int kd = 0; kd < 3; ++kd) {
                    const uint32_t slot = ring_a + (uint32_t)(((s + kd) & (kTfRing - 1)) * SLOT) + (uint32_t)(mt * 128 * 16);
#pragma unroll
                    for (int p = 0; p < NP; ++p) {
                        const int g0 = 2 * p, g1 = 2 * p + 1;
                        const int o0 = (g0 / 9) * kTfSlab + ((g0 % 9) / 3) * Wq + g0 % 3;
                        const int o1 = g1 < 9 * CG ? (g1 / 9) * kTfSlab + ((g1 % 9) / 3) * Wq + g1 % 3 : o0;
                        const uint64_t a = smem_desc(slot + (uint32_t)o0 * 16, (uint32_t)(o1 - o0) * 16, 128);
                        const uint64_t bd = smem_desc(b_a + (uint32_t)((kd * NP + p) * 512), 256, 128);
                        mma_tf32(tmem + (uint32_t)(mt * kTfN), a, bd, acc);
                        acc = 1;
                    }
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
        }
        if (s + 1 < ns) stage(d0 + s + 2, s + 3);                 // the slot plane d-2 used: its MMAs completed last step
        fence_async_smem();
        mbar_wait(bar, (uint32_t)(s & 1));
        fence_after_sync();
        const int d = d0 + s;
#pragma unroll
        for (int mt = 0; mt < kTfRows / 128; ++mt) {
            float v[16];
            tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(mt * kTfN), v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const int q = mt * 128 + tid, row = q / Wq, col = q - row * Wq, h = h0 + row, wo = w0 + col;
            if (row < Ht && col < Wt && h < H && wo < W) {
                float* o = out + (((size_t)b * CO * D + d) * H + h) * W + wo;
#pragma unroll
                for (int c = 0; c < CO; ++c) {
                    float r = scale ? __fmaf_rn(v[c], sc[c], sh[c]) : v[c];
                    if (relu) r = fmaxf(r, 0.f);
                    o[(size_t)c * chan] = r;
                }
            }
        }
        fence_before_sync();
        __syncthreads();                                          // accumulator read, next plane staged
    }
    if (warp == 0) {
        fence_after_sync();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(kTfTmemCols));
    }
}

// ---- host ---------------------------------------------------------------------------------------------------------------
// The patch: the number of column tiles that needs the fewest (CTA, plane) steps; Ht rows of Wt + 2 fill 256 M rows.
static void tf_patch(int H, int W, int& Wt, int& Ht, int& n_wt, int& n_ht) {
    long long best = LLONG_MAX;
    const int n0 = (W + kTfMaxWq - 3) / (kTfMaxWq - 2);
    for (int n = n0; n <= n0 + 3 && n <= W; ++n) {
        const int wt = (W + n - 1) / n, ht = std::min(kTfRows / (wt + 2), H), nh = (H + ht - 1) / ht;
        if ((long long)n * nh < best) { best = (long long)n * nh; Wt = wt; Ht = ht; n_wt = n; n_ht = nh; }
    }
}

template <int CI, int CO, bool FLIP>
static int tf_launch(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                     int B, int D, int H, int W, cudaStream_t st) {
    auto k = conv3d_cc_tf32_kernel<CI, CO, FLIP>;
    const size_t smem = tf_smem(CI);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d_cc_tf32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    int Wt = 0, Ht = 0, n_wt = 0, n_ht = 0;
    tf_patch(H, W, Wt, Ht, n_wt, n_ht);
    const int n_dt = (D + kTfDT - 1) / kTfDT;
    k<<<dim3(n_wt, n_ht, B * n_dt), kTfThreads, smem, st>>>(in, w, scale, shift, relu, out, D, H, W, Wt, Ht, n_dt);
    return check_launch(FLIP ? "conv3d_cc_tf32_bwd_data" : "conv3d_cc_tf32_fwd");
}

int conv3d_cc_tf32_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                       int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!in || !w || !out || (scale == nullptr) != (shift == nullptr))
        return fail(RAG_E_NULL, "conv3d_cc_tf32_fwd: null pointer (scale and shift go together)");
    if (int rc = cc_check("conv3d_cc_tf32_fwd", B, C, O, D, H, W)) return rc;
    if (!aligned(in, 16) || !aligned(out, 16) || !aligned(w, 4)) return fail(RAG_E_ALIGN, "conv3d_cc_tf32_fwd: in/out must be 16-byte aligned");
    switch (C) {
        case 4: return tf_launch<4, 4, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
        case 8: return tf_launch<8, 8, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
        default: return tf_launch<12, 12, false>(in, w, scale, shift, relu, out, B, D, H, W, st);
    }
}

int conv3d_cc_tf32_bwd_data(const float* gz, const float* w, float* gin, int B, int C, int O, int D, int H, int W, cudaStream_t st) {
    if (!gz || !w || !gin) return fail(RAG_E_NULL, "conv3d_cc_tf32_bwd_data: null pointer");
    if (int rc = cc_check("conv3d_cc_tf32_bwd_data", B, C, O, D, H, W)) return rc;
    if (!aligned(gz, 16) || !aligned(gin, 16) || !aligned(w, 4)) return fail(RAG_E_ALIGN, "conv3d_cc_tf32_bwd_data: gz/gin must be 16-byte aligned");
    switch (C) {
        case 4: return tf_launch<4, 4, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st);
        case 8: return tf_launch<8, 8, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st);
        default: return tf_launch<12, 12, true>(gz, w, nullptr, nullptr, 0, gin, B, D, H, W, st);
    }
}

}  // namespace rag
