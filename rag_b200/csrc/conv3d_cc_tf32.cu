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
__global__ void conv3d_cc_wgrad_final_kernel(const float* __restrict__ part, float* __restrict__ gw, int n, int G);   // conv3d_cc.cu

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
// N >> 3 at bits 17-22, M >> 4 at bits 24-28 (M = 128)
__host__ __device__ constexpr uint32_t tf_idesc(int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
constexpr uint32_t kTfIdesc = tf_idesc(kTfN);

template <uint32_t IDESC = kTfIdesc>
__device__ __forceinline__ void mma_tf32(uint32_t dtmem, uint64_t a, uint64_t b, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(dtmem), "l"(a), "l"(b), "r"(IDESC), "r"(accumulate));
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

// ---- weight gradient ----------------------------------------------------------------------------------------------------
// gw[o,c,kd,kh,kw] = sum_{b,d,h,w} gz[b,o,d,h,w] x[b,c,d+kd-1,h+kh-1,w+kw-1] as D[m, n] = sum_k A[m, k] B[k, n] with
// m = a tap row (kh, kw, c), k = an output position along w, and n = (kd, o): the three gz planes around one x plane.
//
// A (x).  A tile is Ht = 4 output rows x Wt = 32 positions of one batch item, walked over every plane.  An x plane of the
// tile is staged as lines h0-1 .. h0+Ht, each as 3C copies (kw, c) shifted by kw - 1 along w (rounded, zero-filled at the
// volume's edges), one 16-byte row per (copy, 4 positions); a line takes R = 3C rounded up to 8 rows (40 / 24 for C = 12 / 8),
// so output row h's 9C tap rows (kh, kw, c) are the one M = 128 range that starts at line h-1: a descriptor offset.  D rows
// past 3R, or on a line's padding, are dropped.  Layout [k-group w/4][row][4]: SBO = 128, LBO = the k-group stride, an odd
// number of 16-byte rows so that staging (8 consecutive k-groups per quarter warp) is free of bank conflicts.
//
// B (gz).  x plane p feeds kd = 0, 1, 2 through gz planes p+1, p, p-1; with those three planes side by side in N
// (n = j*O + o, j = 2 - kd; N = 3*O padded to 16: 48 / 32) one MMA serves all three kd, so A -- the operand that is re-read
// from shared memory for every MMA -- is read once per position instead of three times.  gz planes run through a 4-entry
// ring (a window of three + one staged ahead) of O-row slots per output row and k-group; entries 0 and 1 are also written
// after entry 3 so that every window is 3*O contiguous rows.  The N - 3*O padding columns read past the window (possibly a
// plane being staged) and are never read back.  The stream of gz entries is, per tile, a zero plane and then its D planes;
// a tile takes D + 1 steps (the last issues no MMA) so that each step stages exactly one x plane and one gz entry:
//     step s = (tile k, plane p):  MMAs of x plane p against entries s, s+1, s+2 (gz planes p-1, p, p+1); x planes -1 and
//     D are never staged, gz planes -1 and D are the zero entries.
//
// Pipeline.  One thread issues step s's Ht * Wt/8 MMAs (skipping rows past H and k-steps past W) and commits them; all threads
// wait for step s-1's MMAs (their slots are the ones the next staging overwrites) and stage x plane p+1 and gz entry s+3.
// The accumulator (N columns of TMEM) stays for the CTA's whole walk.  A fixed grid of kTwGroups CTAs takes tiles
// blockIdx.x, blockIdx.x + G, ...; at the end each CTA reads its accumulator once and writes one fp32 partial per sum in
// conv3d_cc.cu's layout [G][O][C][27], and conv3d_cc_wgrad_final_kernel adds them in fp64: bitwise repeatable on any device.
constexpr int kTwHt = 4, kTwWt = 32, kTwKG = kTwWt / 4;   // tile: output rows, positions, 16-byte k-groups per row
constexpr int kTwRing = 4;                                  // gz entries: a window of three + one staged ahead
constexpr int kTwGroups = 296;                              // CTAs (= partials per sum): two per SM of a B200
constexpr int kTwTmemCols = 64;

__host__ __device__ constexpr int tw_line(int C) { return (3 * C + 7) / 8 * 8; }                  // A rows per x line
__host__ __device__ constexpr int tw_akg(int C) { return (((kTwHt - 1) * tw_line(C) + 128) | 1) * 16; }  // bytes per k-group
__host__ __device__ constexpr int tw_n(int O) { return (3 * O + 15) / 16 * 16; }                   // MMA N
__host__ __device__ constexpr int tw_bkg(int O) { return ((3 * O + tw_n(O)) | 1) * 16; }           // window at entry 3 + N rows
__host__ __device__ constexpr size_t tw_smem(int C, int O) {
    return (size_t)2 * kTwKG * tw_akg(C) + (size_t)kTwHt * kTwKG * tw_bkg(O);
}

// grid: G = min(kTwGroups, n_tiles); 128 threads; smem tw_smem(C, O).  part [G][O][C][27].
template <int C, int O>
__global__ void __launch_bounds__(kTfThreads, 2)
conv3d_cc_tf32_wgrad_kernel(const float* __restrict__ gz, const float* __restrict__ in, float* __restrict__ part,
                            int D, int H, int W, int n_ht, int n_wt, int n_tiles) {
    static_assert(C % 4 == 0 && 3 * tw_line(C) <= 128 && tw_n(O) <= 64, "three lines fit one M tile; N fits the TMEM columns");
    constexpr int R = tw_line(C), AKG = tw_akg(C), N = tw_n(O), BKG = tw_bkg(O);
    constexpr int ASLOT = kTwKG * AKG, BROW = kTwKG * BKG;     // bytes of an x slot; of one output row's gz ring
    constexpr size_t SMEM = tw_smem(C, O);
    extern __shared__ __align__(128) unsigned char tf_smem_buf[];
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t tmem_base;
    unsigned char* xs = tf_smem_buf;                  // [slot 2][k-group][AKG / 16 rows][4]
    unsigned char* gs = tf_smem_buf + 2 * ASLOT;      // [output row][k-group][BKG / 16 rows][4]

    const int tid = threadIdx.x, warp = tid >> 5, G = gridDim.x;
    const size_t plane = (size_t)H * W, chan = (size_t)D * plane;
    const int n_local = (n_tiles - (int)blockIdx.x + G - 1) / G;   // >= 1: G <= n_tiles
    const int steps = n_local * (D + 1);                           // < 2^31 (checked on the host)

    // line padding, the rows past the last line and the padding rows of the gz ring are never staged: zero them once
    for (int i = tid; i < (int)(SMEM / 16); i += kTfThreads) reinterpret_cast<float4*>(tf_smem_buf)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_addr(&tmem_base)), "r"(kTwTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(&mbar[0])), "r"(1));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(&mbar[1])), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();                                   // the zero fill is complete before any staging overwrites it

    auto tile_of = [&](int k, int& b, int& h0, int& w0) {
        int t = (int)blockIdx.x + k * G;
        const int wt = t % n_wt;
        t /= n_wt;
        const int ht = t % n_ht;
        b = t / n_ht;
        h0 = ht * kTwHt;
        w0 = wt * kTwWt;
    };
    // Staging is split into loads into registers and stores to shared memory, so that all of a step's loads are in flight
    // at once (and before the wait for the previous step's MMAs) rather than one round trip per item.
    // x plane p of local tile k: per line l and channel c one float4 of positions 4j..4j+3 and its two neighbours give the
    // three shifted copies
    constexpr int NXI = (kTwHt + 2) * C * kTwKG, NX = (NXI + kTfThreads - 1) / kTfThreads;
    constexpr int NGI = kTwHt * O * kTwKG, NG = (NGI + kTfThreads - 1) / kTfThreads;
    float4 xv[NX], gv[NG];
    float xl[NX], xr[NX];
    auto load_x = [&](int k, int p) {
        int b, h0, w0;
        tile_of(k, b, h0, w0);
        const float* xb = in + ((size_t)b * C * D + p) * plane;
#pragma unroll
        for (int it = 0; it < NX; ++it) {
            const int i = tid + it * kTfThreads, j = i % kTwKG, r1 = i / kTwKG, c = r1 % C, l = r1 / C;
            const int gh = h0 - 1 + l, gw = w0 + 4 * j;
            xv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            xl[it] = xr[it] = 0.f;
            if (i < NXI && gh >= 0 && gh < H && gw < W) {   // W % 4 == 0: the float4 is inside the row
                const float* src = xb + (size_t)c * chan + (size_t)gh * W + gw;
                xv[it] = __ldg(reinterpret_cast<const float4*>(src));
                if (gw > 0) xl[it] = __ldg(src - 1);
                if (gw + 4 < W) xr[it] = __ldg(src + 4);
            }
        }
    };
    auto store_x = [&](int sl) {
#pragma unroll
        for (int it = 0; it < NX; ++it) {
            const int i = tid + it * kTfThreads, j = i % kTwKG, r1 = i / kTwKG, c = r1 % C, l = r1 / C;
            if (i < NXI) {
                const float4 v = make_float4(tf32_rna(xv[it].x), tf32_rna(xv[it].y), tf32_rna(xv[it].z), tf32_rna(xv[it].w));
                float4* d = reinterpret_cast<float4*>(xs + sl * ASLOT + j * AKG) + l * R + c;
                d[0] = make_float4(tf32_rna(xl[it]), v.x, v.y, v.z);      // kw = 0: x[w - 1]
                d[C] = v;                                                 // kw = 1
                d[2 * C] = make_float4(v.y, v.z, v.w, tf32_rna(xr[it]));  // kw = 2: x[w + 1]
            }
        }
    };
    // gz entry e: local tile e / (D+1), plane e % (D+1) - 1; plane -1, and every entry past the last tile, is zeros
    auto load_gz = [&](int e) {
        const int k = e / (D + 1), q = e - k * (D + 1) - 1;
        const bool live = q >= 0 && k < n_local;
        int b = 0, h0 = 0, w0 = 0;
        if (live) tile_of(k, b, h0, w0);
        const float* gb = gz + ((size_t)b * O * D + (live ? q : 0)) * plane;
#pragma unroll
        for (int it = 0; it < NG; ++it) {
            const int i = tid + it * kTfThreads, j = i % kTwKG, r1 = i / kTwKG, o = r1 % O, r = r1 / O;
            const int gh = h0 + r, gw = w0 + 4 * j;
            gv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < NGI && live && gh < H && gw < W)
                gv[it] = __ldg(reinterpret_cast<const float4*>(gb + (size_t)o * chan + (size_t)gh * W + gw));
        }
    };
    auto store_gz = [&](int e) {
        const int pos = e % kTwRing;
#pragma unroll
        for (int it = 0; it < NG; ++it) {
            const int i = tid + it * kTfThreads, j = i % kTwKG, r1 = i / kTwKG, o = r1 % O, r = r1 / O;
            if (i < NGI) {
                const float4 v = make_float4(tf32_rna(gv[it].x), tf32_rna(gv[it].y), tf32_rna(gv[it].z), tf32_rna(gv[it].w));
                float4* d = reinterpret_cast<float4*>(gs + r * BROW + j * BKG) + pos * O + o;
                d[0] = v;
                if (pos < 2) d[kTwRing * O] = v;           // the copy that keeps windows starting at entry 2 or 3 contiguous
            }
        }
    };

    load_x(0, 0);
    store_x(0);
    for (int e = 0; e < 3; ++e) {
        load_gz(e);
        store_gz(e);
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tmem_base, xa = smem_addr(xs), ga = smem_addr(gs);

    uint32_t acc = 0;
    int n_commit = 0;                                  // commits before this step: the same count in every thread
    bool prev = false;                                 // step s-1 issued MMAs
#pragma unroll 1
    for (int s = 0; s < steps; ++s) {
        const int k = s / (D + 1), p = s - k * (D + 1);
        const bool mma = p < D;
        if (mma && tid == 0) {
            int b, h0, w0;
            tile_of(k, b, h0, w0);
            const int nr = min(kTwHt, H - h0), nk = (min(kTwWt, W - w0) + 7) / 8;
            const uint32_t a0 = xa + (uint32_t)((s & 1) * ASLOT), b0 = ga + (uint32_t)((s % kTwRing) * O * 16);
            fence_after_sync();
#pragma unroll 1
            for (int r = 0; r < nr; ++r) {
#pragma unroll 1
                for (int kk = 0; kk < nk; ++kk) {
                    const uint64_t a = smem_desc(a0 + (uint32_t)(2 * kk * AKG + r * R * 16), AKG, 128);
                    const uint64_t bd = smem_desc(b0 + (uint32_t)(r * BROW + 2 * kk * BKG), BKG, 128);
                    mma_tf32<tf_idesc(N)>(tmem, a, bd, acc);
                    acc = 1;
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                         :: "r"(smem_addr(&mbar[n_commit & 1])) : "memory");
        }
        const int k1 = (s + 1) / (D + 1), p1 = s + 1 - k1 * (D + 1);
        const bool more = s + 1 < steps, next_x = more && p1 < D;
        if (next_x) load_x(k1, p1);
        if (more) load_gz(s + 3);
        if (prev) {                                    // step s-1's MMAs read the x slot and the gz entry stored below
            const int c = n_commit - 1;
            mbar_wait(smem_addr(&mbar[c & 1]), (uint32_t)((c >> 1) & 1));
        }
        if (mma) ++n_commit;
        prev = mma;
        if (next_x) store_x((s + 1) & 1);
        if (more) store_gz(s + 3);
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        fence_after_sync();
    }
    // the last step issues no MMA and waited for every earlier one: the accumulator is final.  Thread t = TMEM lane t = row t.
    float v[N / 16][16];
#pragma unroll
    for (int i = 0; i < N / 16; ++i) tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(i * 16), v[i]);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const int kh = tid / R, kw = (tid - kh * R) / C, c = tid - kh * R - kw * C;
    if (kh < 3 && kw < 3) {
        float* pp = part + (size_t)blockIdx.x * O * C * 27 + (size_t)c * 27 + kh * 3 + kw;
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int o = 0; o < O; ++o) pp[(size_t)o * C * 27 + (2 - j) * 9] = v[(j * O + o) / 16][(j * O + o) % 16];
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        fence_after_sync();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(kTwTmemCols));
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

static bool tw_pair(int C, int O) { return C == O && (C == 8 || C == 12); }

template <int C, int O>
static int tw_launch(const float* gz, const float* in, float* gw, float* part, int B, int D, int H, int W, int n_tiles,
                     cudaStream_t st) {
    const int n_ht = (H + kTwHt - 1) / kTwHt, n_wt = (W + kTwWt - 1) / kTwWt;
    const int G = std::min(kTwGroups, n_tiles);                   // a function of the shape only: repeatable on any device
    auto k = conv3d_cc_tf32_wgrad_kernel<C, O>;
    const size_t smem = tw_smem(C, O);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d_cc_tf32_bwd_weight: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    k<<<G, kTfThreads, smem, st>>>(gz, in, part, D, H, W, n_ht, n_wt, n_tiles);
    if (int rc = check_launch("conv3d_cc_tf32_bwd_weight")) return rc;
    const int n = O * C * 27;
    conv3d_cc_wgrad_final_kernel<<<(n + 255) / 256, 256, 0, st>>>(part, gw, n, G);
    return check_launch("conv3d_cc_tf32_bwd_weight(final)");
}

size_t conv3d_cc_tf32_bwd_weight_workspace_bytes(int B, int C, int O, int D, int H, int W) {
    if (!tw_pair(C, O) || B <= 0 || D <= 0 || H <= 0 || W <= 0) return 0;
    return (size_t)kTwGroups * O * C * 27 * sizeof(float);
}

int conv3d_cc_tf32_bwd_weight(const float* gz, const float* in, float* gw, float* workspace, int B, int C, int O, int D, int H,
                              int W, cudaStream_t st) {
    if (!gz || !in || !gw || !workspace) return fail(RAG_E_NULL, "conv3d_cc_tf32_bwd_weight: null pointer");
    if (!tw_pair(C, O))
        return fail(RAG_E_SHAPE, "conv3d_cc_tf32_bwd_weight: (C, O) = (%d, %d) is not compiled; have (8,8), (12,12)", C, O);
    if (int rc = cc_check("conv3d_cc_tf32_bwd_weight", B, C, O, D, H, W)) return rc;
    const long long n_tiles = (long long)B * ((H + kTwHt - 1) / kTwHt) * ((W + kTwWt - 1) / kTwWt);
    if (n_tiles * (D + 1) >= (1LL << 31)) return fail(RAG_E_SHAPE, "conv3d_cc_tf32_bwd_weight: too many tiles");
    if (!aligned(gz, 16) || !aligned(in, 16) || !aligned(gw, 4) || !aligned(workspace, 4))
        return fail(RAG_E_ALIGN, "conv3d_cc_tf32_bwd_weight: gz/in must be 16-byte aligned, gw/workspace 4-byte");
    if (C == 8) return tw_launch<8, 8>(gz, in, gw, workspace, B, D, H, W, (int)n_tiles, st);
    return tw_launch<12, 12>(gz, in, gw, workspace, B, D, H, W, (int)n_tiles, st);
}

}  // namespace rag
