/*
 * rag_b200.h -- C ABI of librag_b200.so: the B200 (sm_100a) stereo hot path of chzhang18/RAG.
 *
 * The reference (pure PyTorch) has no FFI for this path; these entry points are what a
 * binding for it would call.  Each one names the reference lines it replaces (paths
 * relative to the reference repo root).  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous row-major fp32 unless it says "host";
 *   - the caller owns every buffer (inputs, outputs, stats); the library never allocates,
 *     frees or retains device memory; outputs are fully overwritten (no pre-zeroing needed);
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream) on the calling thread's current device; no host synchronisation;
 *   - return value: 0 on success; <0 argument error (RAG_E_*); >0 a cudaError_t.  The text
 *     of the last error on the calling thread is rag_last_error().  No exceptions cross the ABI;
 *   - re-entrant and thread-safe.  The library keeps NO mutable state of its own that a launch depends on:
 *     work counters and regrouped weights live in caller-owned workspaces (rag_cost_volume_fwd_ws,
 *     rag_cv_stem_fwd); the thread-local error text and the launch counter are bookkeeping only.  The single
 *     exception is rag_conv3d_c1_fwd, whose weights must sit in constant memory: its eight per-device weight
 *     slots are ordered across streams with events (never rewritten under a running reader) and it refuses a
 *     capturing stream with RAG_E_CAPTURE.  Every other entry point may be stream-captured and the captured
 *     graphs replayed concurrently with eager launches.
 *
 * Shapes: B batch (stereo pairs), C feature channels (12 in the reference), Hf,Wf = H/3,W/3,
 * Df = int(maxdisp/3) low-res disparity bins, D = maxdisp full-res bins.
 */
#ifndef RAG_B200_H
#define RAG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAG_B200_ABI_VERSION 18

#if defined(__GNUC__)
#define RAG_API __attribute__((visibility("default")))
#else
#define RAG_API
#endif

#define RAG_OK 0
#define RAG_E_NULL (-1)     /* a required pointer is NULL                      */
#define RAG_E_SHAPE (-2)    /* a dimension is <= 0 or out of the supported range */
#define RAG_E_ALIGN (-3)    /* a pointer is not 4-byte (16-byte where stated) aligned */
#define RAG_E_VARIANT (-4)  /* unknown kernel variant id                        */
#define RAG_E_CAPTURE (-5)  /* the stream is being captured and this entry point cannot be (rag_conv3d_c1_fwd) */

RAG_API int rag_abi_version(void);
RAG_API const char* rag_last_error(void);
/* Number of kernels this library has launched from the calling process (monotonic counter;
 * used by bench.py to report `gpu_launches`). */
RAG_API uint64_t rag_launch_count(void);

/* ---- cost volume -------------------------------------------------------------------------
 * Replaces src/models/rag_model.py:375-383 (Network.forward), :694-702 (search_forward) and
 * src/automl/mdenas_basicmodel.py:83-91 (BasicNetwork.forward):
 *   cost[b,   c, d,h,w] = x[b,c,h,w]   if w >= d else 0
 *   cost[b, C+c, d,h,w] = y[b,c,h,w-d] if w >= d else 0          d in [0,Df)
 * x,y [B,C,Hf,Wf]; cost [B,2C,Df,Hf,Wf].  Bit-exact copy.  Stateless: one CTA per work item. */
RAG_API int rag_cost_volume_fwd(const float* x, const float* y, float* cost,
                        int B, int C, int Df, int Hf, int Wf, void* stream);
/* Same result through the persistent kernel (one CTA per SM taking its work items IN ORDER from a counter: 3 %
 * faster at B=8 480x960, and the form that can share the SMs with the disparity head on a second stream).
 * workspace: caller-owned DEVICE buffer of RAG_CV_FWD_WORKSPACE_BYTES, 8-byte aligned, private to this launch
 * until it completes; the library zeroes it on `stream` before the kernel (one memset node: graph-capturable).
 * NULL workspace = rag_cost_volume_fwd. */
#define RAG_CV_FWD_WORKSPACE_BYTES 16
RAG_API int rag_cost_volume_fwd_ws(const float* x, const float* y, float* cost,
                           int B, int C, int Df, int Hf, int Wf, void* workspace, void* stream);

/* Gradient of the above (replaces the 128 chained CopySlices autograd nodes the reference
 * loop creates).  gx[b,c,h,w] = sum_d gcost[b,c,d,h,w] (d<=w), gy[b,c,h,w] = sum_d
 * gcost[b,C+c,d,h,w+d] (w+d<Wf); both summed sequentially in fp32 with d DESCENDING, which is
 * the order autograd uses, so the result is bit-identical to the reference.  No atomics. */
RAG_API int rag_cost_volume_bwd(const float* gcost, float* gx, float* gy,
                        int B, int C, int Df, int Hf, int Wf, void* stream);

/* ---- disparity head ----------------------------------------------------------------------
 * Replaces src/models/rag_model.py:32-44 (Disp.forward) + :18-29 (DisparityRegression):
 *   v = trilinear_upsample(cost_lr -> [maxdisp, 3Hl, 3Wl], align_corners=False)
 *   disp[b,h,w] = sum_k k * softmax_k(-v[b,k,h,w])
 * cost_lr [B,1,Dl,Hl,Wl] (Dl need not equal maxdisp/3); disp [B,3Hl,3Wl].
 * stats (nullable) [B,2,3Hl,3Wl]: plane 0 = reference exponent m (log2 domain), plane 1 =
 * 1/sum_k 2^(z_k-m) with z_k = -log2(e)*v_k -- what the backward needs to rebuild p_k. */
RAG_API int rag_disp_head_fwd(const float* cost_lr, float* disp, float* stats,
                      int B, int Dl, int Hl, int Wl, int maxdisp, void* stream);

/* Gradient of the head w.r.t. cost_lr (replaces autograd through interpolate/softmin/mul/sum;
 * PyTorch's CUDA trilinear backward accumulates up to 125 atomicAdds per element in arrival order
 * -- this one is bitwise deterministic: every element of gcost_lr receives exactly TWO contributions,
 * added into the zeroed buffer with red.global.add; two addends commute, so arrival order cannot matter).
 * gdisp, disp [B,3Hl,3Wl]; stats [B,2,3Hl,3Wl] from the forward; gcost_lr [B,1,Dl,Hl,Wl].
 * scratch: may be NULL.  Only the A/B variant 2 of rag_disp_head_bwd_v uses it (a caller-owned
 * work buffer of the same size as gcost_lr, contents undefined on return). */
RAG_API int rag_disp_head_bwd(const float* cost_lr, const float* gdisp, const float* disp,
                      const float* stats, float* gcost_lr, float* scratch,
                      int B, int Dl, int Hl, int Wl, int maxdisp, void* stream);

/* DisparityRegression alone (src/models/rag_model.py:18-29): p [B,D,H,W] -> out [B,H,W],
 * out = sum_k k*p[b,k,h,w]. */
RAG_API int rag_disparity_regression_fwd(const float* p, float* out, int B, int D, int H, int W, void* stream);
/* Its gradient: gp[b,k,h,w] = k * gout[b,h,w]. */
RAG_API int rag_disparity_regression_bwd(const float* gout, float* gp, int B, int D, int H, int W, void* stream);

/* Debug/validation: the upsample alone (F.interpolate at rag_model.py:40), out [B,maxdisp,3Hl,3Wl].
 * fma_index != 0 evaluates the source index with a fused multiply-add (what PyTorch's CUDA
 * kernel compiles to); 0 uses separate multiply and subtract. */
RAG_API int rag_upsample_trilinear(const float* cost_lr, float* out, int B, int Dl, int Hl, int Wl,
                           int maxdisp, int fma_index, void* stream);

/* ---- variants (A/B measurement and fallbacks; the functions above pick the default) ----------
 * Variant ids (-1 = the default; any other id not listed here returns RAG_E_VARIANT):
 *   rag_cost_volume_fwd_v  0 = any width / alignment (items dealt to threads); 1 = lean thread-stationary kernel, one CTA
 *                          per item (default without a workspace when Wf % 4 == 0); 3 = lean persistent, 512 threads (SM
 *                          sharing, launch order); 5 = lean persistent, 256 threads x 1 vector at 48 registers, 32
 *                          disparities per item (default with a workspace; co-resident SM sharing).  3 and 5 need the
 *                          workspace.  Ids 2 (lean persistent, 256 threads x 2 vectors) and 4 (TMA bulk-store kernel) were
 *                          retired in ABI version 18: slower than 5 on every measured shape.
 *   rag_cost_volume_bwd_v  0 = 128-bit vector kernel (default when Wf % 4 == 0), 1 = scalar (any width),
 *                          2 = the vector kernel as a persistent grid of 4 CTAs per SM (SM sharing, launch order);
 *                          3 = cp.async ring in shared memory, one 256-thread CTA per SM at 64 registers (co-resident SM
 *                          sharing)
 *   rag_disp_head_fwd_v    0 = any (Dl, maxdisp); 1 = first x3 kernel (any width); 2 = cube-root tiled kernel (default when
 *                          maxdisp == 3*Dl and Wl % 4 == 0); 4 = 2 as a persistent grid of 3 CTAs per SM (co-resident SM
 *                          sharing).  Id 3 (2 with the lambda correction at every step + TwoSum totals) was retired in ABI
 *                          version 18.
 *   rag_disp_head_bwd_v    0 = any-ratio gather; 1 = block-row tasks, parts added in place (default when maxdisp == 3*Dl);
 *                          2 = same with scratch + combine kernel; 3 = 1 as a persistent grid of 3 CTAs per SM (co-resident)
 *   rag_cv_stem_fwd_v      0 = direct (any shape); 1 = collapsed, scalar; 2 = default (packed phase 1)
 * SM sharing.  The volume kernels are HBM bound and need few issue slots, the head kernels are FP32 bound and need little
 * bandwidth: on two streams they can share the SMs (rag_b200.pipeline).  Two ways:
 *  - launch order (inference): the cost volume is launched FIRST with RAG_CV_FWD_SHARED -- a persistent grid of one
 *    512-thread CTA per SM that is resident at once -- and the head's CTAs are dispatched beside it;
 *  - co-resident (training step; free-running streams cannot control the launch order): ALL four kernels run as persistent
 *    grids whose CTAs fit an SM together -- the volume kernel in a quarter of the register file (RAG_CV_FWD_SLIM: 256 threads
 *    x 48 registers; RAG_CV_BWD_SLIM: 256 threads x 64 registers, its ~96 KB of in-flight reads parked in SHARED memory by
 *    cp.async instead of in registers), three 128-thread x 128-register head CTAs in the rest (RAG_HEAD_FWD_SHARED,
 *    RAG_HEAD_BWD_SHARED) -- so they overlap whichever is launched first.  Every variant gives the same bits as the default. */
#define RAG_CV_FWD_SHARED 3   /* same kernel, one 512-thread CTA per SM: best when launched before the head forward */
#define RAG_CV_FWD_SLIM 5     /* default with a workspace: 256 threads x 1 vector, 32 disparities per item -- a quarter of
                               * the register file (co-resident SM sharing) and the fastest geometry alone as well    */
#define RAG_CV_BWD_SHARED 2   /* backward as a persistent grid: launched first, it leaves room for the head backward */
#define RAG_CV_BWD_SLIM 3     /* backward through a shared-memory cp.async ring: a quarter of the register file     */
#define RAG_HEAD_FWD_SHARED 4 /* head forward as a persistent grid of 3 CTAs per SM                                 */
#define RAG_HEAD_BWD_SHARED 3 /* head backward as a persistent grid of 3 CTAs per SM                                */
RAG_API int rag_cost_volume_fwd_v(const float* x, const float* y, float* cost,
                          int B, int C, int Df, int Hf, int Wf, void* workspace, int variant, void* stream);
RAG_API int rag_cost_volume_bwd_v(const float* gcost, float* gx, float* gy,
                          int B, int C, int Df, int Hf, int Wf, int variant, void* stream);
RAG_API int rag_disp_head_fwd_v(const float* cost_lr, float* disp, float* stats,
                        int B, int Dl, int Hl, int Wl, int maxdisp, int variant, void* stream);
RAG_API int rag_disp_head_bwd_v(const float* cost_lr, const float* gdisp, const float* disp,
                        const float* stats, float* gcost_lr, float* scratch,
                        int B, int Dl, int Hl, int Wl, int maxdisp, int variant, void* stream);

/* ---- adjacent rows (SURVEY.md section 8f) -------------------------------------------------
 * Masked loss + metrics on the disparity map, one fused reduction.  Replaces
 * src/approaches/rag.py:418-430 + src/utilstool/metrics.py:22-65 (about 10*B tiny kernels and
 * 6+ .item() syncs per batch).  est, gt [B,H,W]; sums: DOUBLE [B,8] per image:
 *   0 n_mask (0<gt<maxdisp)  1 n_pos (gt>0)  2 sum smooth_l1  3 sum |gt-est|
 *   4 n_d1 (E>3 && E/|gt|>0.05)  5 n_E>1  6 n_E>2  7 n_E>3
 * Deterministic (fixed-order reduction, no float atomics).  scratch: DOUBLE [B, rag_loss_metrics_scratch(H,W)]. */
RAG_API int rag_loss_metrics_scratch(int H, int W);
RAG_API int rag_loss_metrics_sums(const float* est, const float* gt, double* sums, double* scratch,
                          int B, int H, int W, float maxdisp, void* stream);
/* gradient of mean masked smooth-L1 (beta=1) w.r.t. est: gest = gloss * dsl1(est-gt) / n_mask_total
 * where mask true, else 0.  n_mask_total read from device `sums` rows (sum over b of sums[b][0]). */
RAG_API int rag_smooth_l1_bwd(const float* est, const float* gt, const double* sums, const float* gloss,
                      float* gest, int B, int H, int W, float maxdisp, void* stream);

/* Fused cost volume + first Matching-Net convolution (inference): the volume is never materialised.
 * Replaces src/models/rag_model.py:375-383 followed by `self.stem3d0[i](cost)` (rag_model.py:341), i.e.
 * ConvBR_3d(2C -> O, 3x3x3, stride 1, pad 1) of src/automl/operations_3d.py:31-47:
 *   out = relu?( scale[o] * conv3d(cost_volume(x, y), w)[o] + shift[o] )
 * x,y [B,C,Hf,Wf]; w [O,2C,3,3,3] (Conv3d.weight, bias-free); scale/shift [O] = eval-mode BatchNorm folded
 * (gamma/sqrt(var+eps), beta - mean*scale), NULL = identity; out [B,O,Df,Hf,Wf].  fp32 accumulation
 * (cuDNN's default for this layer is TF32).
 * workspace (nullable): caller-owned DEVICE buffer of rag_cv_stem_workspace_bytes(C, O) bytes, 16-byte aligned, private
 * to this launch until it completes; the weights are regrouped into it once per launch instead of by every CTA. */
RAG_API size_t rag_cv_stem_workspace_bytes(int C, int O);
RAG_API int rag_cv_stem_fwd(const float* x, const float* y, const float* w, const float* scale, const float* shift,
                    int relu, float* out, int B, int C, int O, int Df, int Hf, int Wf, void* workspace, void* stream);
RAG_API int rag_cv_stem_fwd_v(const float* x, const float* y, const float* w, const float* scale, const float* shift,
                      int relu, float* out, int B, int C, int O, int Df, int Hf, int Wf, void* workspace, int variant, void* stream);

/* Batch statistics of that convolution for a training-mode BatchNorm3d, again without the volume or the conv
 * output (first piece of the training path, DESIGN.md section 10): moments [B,Hf,O,2] DOUBLE, per (b,h,o) row
 * (sum z, sum z^2) over its Df x Wf outputs z = conv3d(cost_volume(x, y), w)[b,o,:,h,:]; the caller sums the rows
 * (mean = S1/n, biased var = S2/n - mean^2, n = B*Df*Hf*Wf).  Needs C == 12, Df >= 3, Wf % 4 == 0.
 * workspace: as for rag_cv_stem_fwd (nullable). */
RAG_API int rag_cv_stem_moments(const float* x, const float* y, const float* w, double* moments,
                        int B, int C, int O, int Df, int Hf, int Wf, void* workspace, void* stream);

/* ---- training-mode BatchNorm3d + ReLU -----------------------------------------------------------------------------------
 * The BatchNorm half of ConvBR_3d (src/automl/operations_3d.py:31-47) in the training paths of the fused stem and of the
 * interior layers, on the convolution output z [B,O,D,H,W], for BatchNorm in train() (batch statistics) or eval() (running
 * statistics).  n = B*D*H*W; bn [O,4] = (scale, shift, mean, rstd) fp32, scale = gamma*rstd, shift = beta - mean*scale.
 * Forward:
 *   rag_bn3d_moments: sums [O,2] DOUBLE = (sum z, sum z^2);
 *   rag_bn3d_finalize: bn from sums (batch != 0: mean, biased variance) or from the running statistics (batch == 0; sums may
 *     be NULL); with batch and update != 0 the running estimates move in place as nn.BatchNorm's do in train()
 *     (r = (1-momentum) r + momentum * batch value, unbiased variance n/(n-1));
 *   rag_bn3d_relu: z <- max(fma(z, scale[o], shift[o]), 0) IN PLACE = the layer output.
 * Backward, with g [B,O,D,H,W] the upstream gradient of the layer output, g' = g [fma(z, scale, shift) > 0] (the forward's own
 * ReLU decision, bit for bit) and zh = (z - mean)*rstd:
 *   rag_bn3d_bwd_sums: sums [O,2] DOUBLE = (sum g', sum g'*zh);
 *   rag_bn3d_bwd_consts: consts [O,7] = (a, m1, m2, scale, shift, mean, rstd) with a = gamma*rstd and, when batch != 0,
 *     m1 = sums[o,0]/n, m2 = sums[o,1]/n, else m1 = m2 = 0; gparam [2,O] = (d/d gamma, d/d beta);
 *   rag_bn3d_bwd_gz: gz [B,O,D,H,W] = a (g' - m1 - zh m2), the gradient at the convolution output.
 * rows_ws: caller-owned DOUBLE workspace [B*H*O*2].  The entry points that take a [B,O,D,H,W] tensor need O <= 32, D >= 3,
 * 8 <= W <= 1016, W % 4 == 0, B <= 32767, H <= 65535 and 16-byte aligned z / g / gz.  Deterministic (fixed-order reductions,
 * no atomics). */
RAG_API int rag_bn3d_moments(const float* z, double* sums, double* rows_ws, int B, int O, int D, int H, int W, void* stream);
RAG_API int rag_bn3d_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                      float* bn, int O, double n, double eps, double momentum, int batch, int update, void* stream);
RAG_API int rag_bn3d_relu(float* z, const float* bn, int B, int O, int D, int H, int W, void* stream);
RAG_API int rag_bn3d_bwd_sums(const float* g, const float* z, const float* bn, double* sums, double* rows_ws,
                      int B, int O, int D, int H, int W, void* stream);
RAG_API int rag_bn3d_bwd_consts(const double* sums, const float* bn, float* consts, float* gparam, int O, double n, int batch, void* stream);
RAG_API int rag_bn3d_bwd_gz(const float* g, const float* z, const float* consts, float* gz, int B, int O, int D, int H, int W, void* stream);

/* The fused layer with autograd (training; DESIGN.md section 5.7) -- again without the volume, its gradient, or any other
 * [B,2C,Df,Hf,Wf] tensor.  Replaces src/models/rag_model.py:375-383 + ConvBR_3d and their autograd.
 * Forward:  z = rag_cv_stem_fwd(x, y, w, NULL, NULL, 0, ...), then the BatchNorm3d forward above: z becomes the layer output.
 * Backward: z is RECOMPUTED with rag_cv_stem_fwd; rag_bn3d_bwd_sums + rag_bn3d_bwd_consts give consts [O,7]; rag_cv_stem_bwd
 *   forms gz on the fly and reduces it along d into 2-D maps, then gx, gy [B,C,Hf,Wf] (both or neither; need w) and
 *   gw [O,2C,3,3,3] (nullable; needs x, y) are 2-D contractions.
 * workspace: rag_cv_stem_bwd_workspace_bytes(B,C,O,Hf,Wf) bytes, 16-byte aligned, caller-owned.  Deterministic (fixed-order
 * reductions, no atomics).  Needs C == 12, O <= 32, Df >= 3, 8 <= Wf <= 1016, Wf % 4 == 0. */
RAG_API size_t rag_cv_stem_bwd_workspace_bytes(int B, int C, int O, int Hf, int Wf);
RAG_API int rag_cv_stem_bwd(const float* g, const float* z, const float* consts, const float* x, const float* y, const float* w,
                    float* gx, float* gy, float* gw, void* workspace, int B, int C, int O, int Df, int Hf, int Wf, void* stream);

/* The Matching Net's last layer, the producer of the head's input (inference):
 * `self.last_3_3d[i](...)` = ConvBR_3d(C, 1, 3, 1, 1, bn=False, relu=False), src/models/rag_model.py:269,361-365,
 * i.e. a bias-free Conv3d C -> 1, 3x3x3, stride 1, zero padding 1 (src/automl/operations_3d.py:31-47):
 *   out[b,0,d,h,w] = sum_{c,kd,kh,kw} w[0,c,kd,kh,kw] * in[b,c,d+kd-1,h+kh-1,w+kw-1]
 * in [B,C,D,H,W]; w [1,C,3,3,3] (Conv3d.weight); out [B,1,D,H,W].  fp32 accumulation (cuDNN's default for
 * this layer is TF32).  Needs W % 4 == 0, C <= 64, B*ceil(D/16) <= 65535 and 16-byte aligned in/out.
 * Not capturable (RAG_E_CAPTURE on a capturing stream): see the conventions at the top of this file. */
RAG_API int rag_conv3d_c1_fwd(const float* in, const float* w, float* out, int B, int C, int D, int H, int W, void* stream);

/* Backward of that layer (training).  g [B,1,D,H,W] = upstream gradient of the layer output.
 *   gin [B,C,D,H,W] (nullable; needs w):  gin[b,c,p] = sum_k w[0,c,k] * g[b,0,p-k+1]
 *   gw  [1,C,3,3,3] (nullable; needs in and workspace):  gw[0,c,k] = sum_{b,p} in[b,c,p+k-1] * g[b,0,p]
 * workspace: rag_conv3d_c1_bwd_workspace_bytes(C) bytes, caller-owned.  Deterministic (fixed-order reductions, no atomics).
 * Needs W % 4 == 0 and 16-byte aligned g / in / gin.  Capturable (weights are read from global memory here). */
RAG_API size_t rag_conv3d_c1_bwd_workspace_bytes(int C);
RAG_API int rag_conv3d_c1_bwd(const float* g, const float* in, const float* w, float* gin, float* gw, void* workspace,
                      int B, int C, int D, int H, int W, void* stream);

/* The Matching Net's interior 3x3x3 layers: ConvBR_3d(C, O, 3, 1, 1) of src/automl/operations_3d.py:31-47 = bias-free
 * Conv3d C -> O (3x3x3, stride 1, zero padding 1) + BatchNorm3d + ReLU -- `stem3d1` (12 -> 12, src/models/rag_model.py) and
 * the `conv_3x3` ops of the Cell_3d's.  Compiled for (C, O) in {(4,4), (8,8), (12,12)}; any other pair is RAG_E_SHAPE.  fp32 accumulation (cuDNN's default for these layers is TF32).  Stateless and capturable.
 * Forward:  out[b,o,p] = relu?( fma(z[b,o,p], scale[o], shift[o]) ),  z[b,o,p] = sum_{c,k} w[o,c,k] in[b,c,p+k-1]
 *   in [B,C,D,H,W]; w [O,C,3,3,3] (Conv3d.weight); scale / shift [O] (both NULL = identity: raw z, the training path;
 *   eval-mode BatchNorm folded: scale = gamma/sqrt(var+eps), shift = beta - mean*scale); relu != 0 clamps at 0;
 *   out [B,O,D,H,W].  Needs W % 4 == 0, 3*H*W < 2^31, B*ceil(D/8) <= 65535, 16-byte aligned in / out.
 * Training: z = the raw forward output (scale = shift = NULL, relu = 0) goes through the BatchNorm3d section above, whose
 * rag_bn3d_bwd_gz gives the gradient gz at the convolution output.
 * rag_conv3d_cc_bwd, from gz:
 *   gin [B,C,D,H,W] (nullable; needs w):            gin[b,c,p] = sum_{o,k} w[o,c,k] gz[b,o,p-k+1]
 *   gw  [O,C,3,3,3] (nullable; needs in, workspace): gw[o,c,k]  = sum_{b,p} gz[b,o,p] in[b,c,p+k-1]
 *   workspace: rag_conv3d_cc_bwd_workspace_bytes(B,C,O,D,H,W) bytes (0 = unsupported pair), caller-owned.  Bitwise
 *   repeatable: fixed-order per-CTA partials, fp64 final pass, no atomics.  Same shape limits as the forward. */
RAG_API int rag_conv3d_cc_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                      int B, int C, int O, int D, int H, int W, void* stream);
RAG_API size_t rag_conv3d_cc_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W);
RAG_API int rag_conv3d_cc_bwd(const float* gz, const float* in, const float* w, float* gin, float* gw, void* workspace,
                      int B, int C, int O, int D, int H, int W, void* stream);

/* The level-12 op, (C, O) = (16, 16), on a small-volume geometry (csrc/conv3d_cc.cu): the arguments, results, limits and
 * errors of rag_conv3d_cc_fwd / rag_conv3d_cc_bwd, compiled for (16,16) only -- any other pair is RAG_E_SHAPE -- plus a
 * weight-gradient tile count B*D*ceil(H/2)*ceil(W/32) < 2^31.  fp32, stateless, capturable; the weight gradient is fixed-order
 * per-CTA partials added in fp64, no atomics: the same bits on any device.  workspace:
 * rag_conv3d_cc16_bwd_workspace_bytes(B,C,O,D,H,W) bytes (0 = unsupported pair; needs no device), caller-owned. */
RAG_API int rag_conv3d_cc16_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                        int B, int C, int O, int D, int H, int W, void* stream);
RAG_API size_t rag_conv3d_cc16_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W);
RAG_API int rag_conv3d_cc16_bwd(const float* gz, const float* in, const float* w, float* gin, float* gw, void* workspace,
                        int B, int C, int O, int D, int H, int W, void* stream);

/* The same layers on the tensor cores in TF32 (csrc/conv3d_cc_tf32.cu): tcgen05.mma kind::tf32, both operands rounded to
 * TF32 with round-to-nearest (ties away) and summed in fp32 -- the precision cuDNN uses for these convolutions by default.
 * Same pairs, arguments, limits and errors as rag_conv3d_cc_fwd / the gin half of rag_conv3d_cc_bwd; stateless, capturable,
 * bitwise repeatable.
 *   rag_conv3d_cc_tf32_fwd:      out = relu?( fma(z, scale, shift) ), z = the forward convolution of in by w.
 *   rag_conv3d_cc_tf32_bwd_data: gin[b,c,p] = sum_{o,k} w[o,c,k] gz[b,o,p-k+1]  (gz [B,O,D,H,W], gin [B,C,D,H,W]).
 *   rag_conv3d_cc_tf32_bwd_weight: gw[o,c,k] = sum_{b,p} gz[b,o,p] in[b,c,p+k-1]  (gw [O,C,3,3,3]), compiled for (8,8) and
 *     (12,12) only: any other pair, (4,4) included, is RAG_E_SHAPE.  Otherwise the arguments, limits and errors of the gw half
 *     of rag_conv3d_cc_bwd; gz / in 16-byte aligned, gw / workspace 4-byte.  workspace:
 *     rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(B,C,O,D,H,W) bytes (0 = unsupported pair; needs no device),
 *     caller-owned.  Fixed-order per-CTA partials added in fp64, no atomics: the same bits on any device. */
RAG_API int rag_conv3d_cc_tf32_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                           int B, int C, int O, int D, int H, int W, void* stream);
RAG_API int rag_conv3d_cc_tf32_bwd_data(const float* gz, const float* w, float* gin, int B, int C, int O, int D, int H, int W, void* stream);
RAG_API size_t rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(int B, int C, int O, int D, int H, int W);
RAG_API int rag_conv3d_cc_tf32_bwd_weight(const float* gz, const float* in, float* gw, void* workspace, int B, int C, int O, int D,
                                  int H, int W, void* stream);

/* The Matching Net's pointwise layers: ConvBR_3d(C, O, 1, 1, 0) of src/automl/operations_3d.py:31-47 = bias-free Conv3d
 * C -> O (1x1x1) + BatchNorm3d + ReLU -- `last_12_3d` (48 -> 24) and `last_6_3d` (24 -> 12) of src/models/rag_model.py.
 * Any (C, O) with 1 <= C <= 64 and 1 <= O <= 32 at run time; fp32 accumulation over c = 0..C-1 in order (cuDNN's default
 * for these layers is TF32).  Stateless and capturable.  S = D*H*W.
 * Forward:  out[b,o,s] = relu?( fma(z[b,o,s], scale[o], shift[o]) ),  z[b,o,s] = sum_c w[o,c] in[b,c,s]
 *   in [B,C,D,H,W]; w [O,C,1,1,1] (Conv3d.weight); scale / shift [O] (both NULL = identity: raw z, the training path;
 *   eval-mode BatchNorm folded: scale = gamma/sqrt(var+eps), shift = beta - mean*scale); relu != 0 clamps at 0;
 *   out [B,O,D,H,W].  Reads in once, writes out once.
 * Training: z = the raw forward output goes through the BatchNorm3d section above; rag_bn3d_bwd_sums + rag_bn3d_bwd_consts give
 * consts [O,7].  rag_conv3d_pw_bwd, from g [B,O,D,H,W] (upstream gradient of the layer output), z and consts, forms the
 * gradient at the convolution output gz = a (g' - m1 - zh m2) on the fly -- the expression of rag_bn3d_bwd_gz, bit for bit --
 * without writing it, and from it:
 *   gin [B,C,D,H,W] (nullable; needs w):            gin[b,c,s] = sum_o w[o,c] gz[b,o,s]
 *   gw  [O,C,1,1,1] (nullable; needs in, workspace): gw[o,c]    = sum_{b,s} gz[b,o,s] in[b,c,s]
 *   workspace: rag_conv3d_pw_bwd_workspace_bytes(B,C,O,D,H,W) bytes (0 = outside the limits), caller-owned.  Bitwise
 *   repeatable: fixed-order per-CTA partials of a fixed grid, fp64 final pass, no atomics.
 * Needs 1 <= C <= 64, 1 <= O <= 32, B <= 65535, S % 4 == 0 and 16-byte aligned in / out / g / z / gin. */
RAG_API int rag_conv3d_pw_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                      int B, int C, int O, int D, int H, int W, void* stream);
RAG_API size_t rag_conv3d_pw_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W);
RAG_API int rag_conv3d_pw_bwd(const float* g, const float* z, const float* consts, const float* in, const float* w, float* gin,
                      float* gw, void* workspace, int B, int C, int O, int D, int H, int W, void* stream);

/* Trilinear resize of [B*C, Di,Hi,Wi] -> [B*C, Do,Ho,Wo] with PyTorch's fp32 index arithmetic: the `upsample_6` /
 * `upsample_12` steps of the Matching Net's tail, nn.Upsample(size=..., mode='trilinear', align_corners=True) at
 * src/models/rag_model.py:356-366 and :675-685 (align_corners = 0 gives F.interpolate's default convention).
 * The backward is a GATHER per input voxel in a fixed order: bitwise repeatable, unlike ATen's atomicAdd scatter. */
RAG_API int rag_trilinear_resize_fwd(const float* in, float* out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                             int align_corners, void* stream);
RAG_API int rag_trilinear_resize_bwd(const float* gout, float* gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo,
                             int align_corners, void* stream);

/* Bilinear resize of [B*C, Hi,Wi] -> [B*C, Ho,Wo]: F.interpolate(..., mode='bilinear') on an NCHW tensor, with the same fp32
 * index arithmetic, argument checks and error codes as the trilinear pair above (the same kernels with the depth axis
 * compiled out).  The backward is a fixed-order gather per input pixel: bitwise repeatable.  Nothing is allocated. */
RAG_API int rag_bilinear_resize_fwd(const float* in, float* out, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners,
                            void* stream);
RAG_API int rag_bilinear_resize_bwd(const float* gout, float* gin, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners,
                            void* stream);

/* 4-D bilinear grid sampling: F.grid_sample(input, grid, mode='bilinear', padding_mode=..., align_corners=...), the warp that
 * synthesises one view from the other and a predicted disparity in the self-supervised loss (src_self/models/loss.py; that the
 * warp is F.grid_sample is inferred, the reference's loss is unread).  Contract: ATen's grid_sampler_2d with its fp32 index
 * arithmetic (csrc/grid_sample.cu states it).  in [N,C,Hi,Wi]; grid [N,Ho,Wo,2] (x, y in [-1, 1]); out [N,C,Ho,Wo].
 * padding_mode: 0 = 'zeros', 1 = 'border' (anything else RAG_E_SHAPE); align_corners: 0 / 1.  grid and ggrid 8-byte aligned.
 * Sizes: 4*N*Ho*Wo, N*Hi*Wi, N*C*Hi*Wi and N*C*Ho*Wo must be below 2^31 (RAG_E_SHAPE, checked on the host).  A grid value of
 * any size, NaN or infinite, reads nothing out of bounds.  Stateless and capturable.
 * rag_grid_sample_bwd, from gout [N,C,Ho,Wo]:
 *   ggrid [N,Ho,Wo,2] (nullable; needs in): ATen's grid gradient, per sample over the channels in ascending order;
 *   gin [N,C,Hi,Wi] (nullable; needs workspace): gin[n,c,y,x] = sum of w * gout[n,c,ho,wo] over every (sample, corner) that reads
 *     (y, x), in ascending flat sample index (n*Ho + ho)*Wo + wo and within a sample in the corner order nw, ne, sw, se --
 *     a fixed order, so the result is bitwise repeatable (ATen's backward adds with atomicAdd in arrival order).  No float atomics.
 * workspace: caller-owned DEVICE buffer of rag_grid_sample_bwd_workspace_bytes(N,C,Hi,Wi,Ho,Wo) bytes (0 = outside the limits),
 *   256-byte aligned, contents undefined on return; workspace_bytes is its size (a smaller one is RAG_E_SHAPE).  It holds 20 bytes
 *   per sample-corner (4*N*Ho*Wo of them: sort keys and values, each double-buffered, and a weight), 8 bytes per input pixel
 *   (N*Hi*Wi segment bounds) and the radix sort's own storage (a few KB); each region rounded up to 256 bytes.  The query needs
 *   no device.  Not needed (may be NULL) when gin is NULL. */
RAG_API int rag_grid_sample_fwd(const float* in, const float* grid, float* out, int N, int C, int Hi, int Wi, int Ho, int Wo,
                        int padding_mode, int align_corners, void* stream);
RAG_API size_t rag_grid_sample_bwd_workspace_bytes(int N, int C, int Hi, int Wi, int Ho, int Wo);
RAG_API int rag_grid_sample_bwd(const float* gout, const float* in, const float* grid, float* gin, float* ggrid, void* workspace,
                        size_t workspace_bytes, int N, int C, int Hi, int Wi, int Ho, int Wo, int padding_mode, int align_corners,
                        void* stream);

/* Eval-time input staging: uint8 HWC image -> ImageNet-normalised fp32 CHW, zero-padded on the
 * top and right.  Replaces src/dataloaders/data_io.py:6-13 + stereo_dataset.py:88-102.
 * img [B,H,W,3] uint8; out [B,3,H+top_pad,W+right_pad] fp32. */
RAG_API int rag_normalize_pad(const uint8_t* img, float* out, int B, int H, int W,
                      int top_pad, int right_pad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAG_B200_H */
