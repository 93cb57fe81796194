// extern "C" surface of librag_b200.so -- see include/rag_b200.h for the contract.
#include "common.cuh"

namespace rag {
thread_local char g_last_error[512] = "";
std::atomic<uint64_t> g_launches{0};

int cost_volume_fwd(const float*, const float*, float*, int, int, int, int, int, void*, int, cudaStream_t);
int cost_volume_bwd(const float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int upsample_trilinear(const float*, float*, int, int, int, int, int, int, cudaStream_t);
int disp_head_fwd(const float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int disp_head_bwd(const float*, const float*, const float*, const float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int disparity_regression_fwd(const float*, float*, int, int, int, int, cudaStream_t);
int disparity_regression_bwd(const float*, float*, int, int, int, int, cudaStream_t);
int loss_metrics_scratch(int, int);
int loss_metrics_sums(const float*, const float*, double*, double*, int, int, int, float, cudaStream_t);
int smooth_l1_bwd(const float*, const float*, const double*, const float*, float*, int, int, int, float, cudaStream_t);
int normalize_pad(const uint8_t*, float*, int, int, int, int, int, cudaStream_t);
int cv_stem_fwd(const float*, const float*, const float*, const float*, const float*, int, float*, int, int, int, int, int, int, float*, int, cudaStream_t);
size_t cv_stem_workspace_bytes(int, int);
int cv_stem_moments(const float*, const float*, const float*, double*, int, int, int, int, int, int, float*, cudaStream_t);
int conv3d_c1_fwd(const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
int conv3d_c1_bwd(const float*, const float*, const float*, float*, float*, float*, int, int, int, int, int, cudaStream_t);
size_t conv3d_c1_bwd_workspace_bytes(int);
int trilinear_resize_fwd(const float*, float*, int, int, int, int, int, int, int, int, cudaStream_t);
int trilinear_resize_bwd(const float*, float*, int, int, int, int, int, int, int, int, cudaStream_t);
int bilinear_resize_fwd(const float*, float*, int, int, int, int, int, int, cudaStream_t);
int bilinear_resize_bwd(const float*, float*, int, int, int, int, int, int, cudaStream_t);
int bn3d_moments(const float*, double*, double*, int, int, int, int, int, cudaStream_t);
int bn3d_finalize(const double*, const float*, const float*, float*, float*, float*, int, double, double, double, int, int, cudaStream_t);
int bn3d_relu(float*, const float*, int, int, int, int, int, cudaStream_t);
int bn3d_bwd_sums(const float*, const float*, const float*, double*, double*, int, int, int, int, int, cudaStream_t);
int bn3d_bwd_consts(const double*, const float*, float*, float*, int, double, int, cudaStream_t);
int bn3d_bwd_gz(const float*, const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
size_t cv_stem_bwd_workspace_bytes(int, int, int, int, int);
int cv_stem_bwd(const float*, const float*, const float*, const float*, const float*, const float*, float*, float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int conv3d_cc_fwd(const float*, const float*, const float*, const float*, int, float*, int, int, int, int, int, int, cudaStream_t);
size_t conv3d_cc_bwd_workspace_bytes(int, int, int, int, int, int);
int conv3d_cc_bwd(const float*, const float*, const float*, float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int conv3d_pw_fwd(const float*, const float*, const float*, const float*, int, float*, int, int, int, int, int, int, cudaStream_t);
size_t conv3d_pw_bwd_workspace_bytes(int, int, int, int, int, int);
int conv3d_pw_bwd(const float*, const float*, const float*, const float*, const float*, float*, float*, float*, int, int, int, int, int, int, cudaStream_t);
int grid_sample_fwd(const float*, const float*, float*, int, int, int, int, int, int, int, int, cudaStream_t);
size_t grid_sample_bwd_workspace_bytes(int, int, int, int, int, int);
int grid_sample_bwd(const float*, const float*, const float*, float*, float*, void*, size_t, int, int, int, int, int, int, int, int, cudaStream_t);
}  // namespace rag

using namespace rag;
#define ST(s) static_cast<cudaStream_t>(s)

// default variants (picked from the measurements in profiles/)
static constexpr int kCvFwdDefault = -1;    // -1 = lean kernel when Wf % 4 == 0 and pointers are 16-byte aligned (persistent with a workspace), cv_fwd_kernel otherwise
static constexpr int kCvBwdDefault = 0;
static constexpr int kHeadFwdDefault = -1;  // -1 = x3 kernel when maxdisp == 3*Dl, generic otherwise
static constexpr int kHeadBwdDefault = -1;

extern "C" {

RAG_API int rag_abi_version(void) { return RAG_B200_ABI_VERSION; }
RAG_API const char* rag_last_error(void) { return g_last_error; }
RAG_API uint64_t rag_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

RAG_API int rag_cost_volume_fwd(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf, void* stream) {
    return cost_volume_fwd(x, y, cost, B, C, Df, Hf, Wf, nullptr, kCvFwdDefault, ST(stream));
}
RAG_API int rag_cost_volume_fwd_ws(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf, void* workspace, void* stream) {
    return cost_volume_fwd(x, y, cost, B, C, Df, Hf, Wf, workspace, kCvFwdDefault, ST(stream));
}
RAG_API int rag_cost_volume_bwd(const float* gcost, float* gx, float* gy, int B, int C, int Df, int Hf, int Wf, void* stream) {
    return cost_volume_bwd(gcost, gx, gy, B, C, Df, Hf, Wf, kCvBwdDefault, ST(stream));
}
RAG_API int rag_disp_head_fwd(const float* cost_lr, float* disp, float* stats, int B, int Dl, int Hl, int Wl, int maxdisp, void* stream) {
    return disp_head_fwd(cost_lr, disp, stats, B, Dl, Hl, Wl, maxdisp, kHeadFwdDefault, ST(stream));
}
RAG_API int rag_disp_head_bwd(const float* cost_lr, const float* gdisp, const float* disp, const float* stats, float* gcost_lr,
                      float* scratch, int B, int Dl, int Hl, int Wl, int maxdisp, void* stream) {
    return disp_head_bwd(cost_lr, gdisp, disp, stats, gcost_lr, scratch, B, Dl, Hl, Wl, maxdisp, kHeadBwdDefault, ST(stream));
}
RAG_API int rag_disparity_regression_fwd(const float* p, float* out, int B, int D, int H, int W, void* stream) {
    return disparity_regression_fwd(p, out, B, D, H, W, ST(stream));
}
RAG_API int rag_disparity_regression_bwd(const float* gout, float* gp, int B, int D, int H, int W, void* stream) {
    return disparity_regression_bwd(gout, gp, B, D, H, W, ST(stream));
}
RAG_API int rag_upsample_trilinear(const float* cost_lr, float* out, int B, int Dl, int Hl, int Wl, int maxdisp, int fma_index, void* stream) {
    return upsample_trilinear(cost_lr, out, B, Dl, Hl, Wl, maxdisp, fma_index, ST(stream));
}

RAG_API int rag_cost_volume_fwd_v(const float* x, const float* y, float* cost, int B, int C, int Df, int Hf, int Wf, void* workspace, int variant, void* stream) {
    return cost_volume_fwd(x, y, cost, B, C, Df, Hf, Wf, workspace, variant, ST(stream));
}
RAG_API int rag_cost_volume_bwd_v(const float* gcost, float* gx, float* gy, int B, int C, int Df, int Hf, int Wf, int variant, void* stream) {
    return cost_volume_bwd(gcost, gx, gy, B, C, Df, Hf, Wf, variant, ST(stream));
}
RAG_API int rag_disp_head_fwd_v(const float* cost_lr, float* disp, float* stats, int B, int Dl, int Hl, int Wl, int maxdisp, int variant, void* stream) {
    return disp_head_fwd(cost_lr, disp, stats, B, Dl, Hl, Wl, maxdisp, variant, ST(stream));
}
RAG_API int rag_disp_head_bwd_v(const float* cost_lr, const float* gdisp, const float* disp, const float* stats, float* gcost_lr,
                        float* scratch, int B, int Dl, int Hl, int Wl, int maxdisp, int variant, void* stream) {
    return disp_head_bwd(cost_lr, gdisp, disp, stats, gcost_lr, scratch, B, Dl, Hl, Wl, maxdisp, variant, ST(stream));
}

RAG_API int rag_loss_metrics_scratch(int H, int W) { return loss_metrics_scratch(H, W); }
RAG_API int rag_loss_metrics_sums(const float* est, const float* gt, double* sums, double* scratch, int B, int H, int W, float maxdisp, void* stream) {
    return loss_metrics_sums(est, gt, sums, scratch, B, H, W, maxdisp, ST(stream));
}
RAG_API int rag_smooth_l1_bwd(const float* est, const float* gt, const double* sums, const float* gloss, float* gest,
                      int B, int H, int W, float maxdisp, void* stream) {
    return smooth_l1_bwd(est, gt, sums, gloss, gest, B, H, W, maxdisp, ST(stream));
}
RAG_API size_t rag_cv_stem_workspace_bytes(int C, int O) { return cv_stem_workspace_bytes(C, O); }
RAG_API int rag_cv_stem_fwd(const float* x, const float* y, const float* w, const float* scale, const float* shift,
                    int relu, float* out, int B, int C, int O, int Df, int Hf, int Wf, void* workspace, void* stream) {
    return cv_stem_fwd(x, y, w, scale, shift, relu, out, B, C, O, Df, Hf, Wf, static_cast<float*>(workspace), -1, ST(stream));
}
RAG_API int rag_cv_stem_moments(const float* x, const float* y, const float* w, double* moments, int B, int C, int O, int Df, int Hf, int Wf,
                        void* workspace, void* stream) {
    return cv_stem_moments(x, y, w, moments, B, C, O, Df, Hf, Wf, static_cast<float*>(workspace), ST(stream));
}
RAG_API int rag_cv_stem_fwd_v(const float* x, const float* y, const float* w, const float* scale, const float* shift,
                      int relu, float* out, int B, int C, int O, int Df, int Hf, int Wf, void* workspace, int variant, void* stream) {
    return cv_stem_fwd(x, y, w, scale, shift, relu, out, B, C, O, Df, Hf, Wf, static_cast<float*>(workspace), variant, ST(stream));
}
RAG_API size_t rag_cv_stem_bwd_workspace_bytes(int B, int C, int O, int Hf, int Wf) { return cv_stem_bwd_workspace_bytes(B, C, O, Hf, Wf); }
RAG_API int rag_cv_stem_bwd(const float* g, const float* pre, const float* consts, const float* x, const float* y, const float* w,
                    float* gx, float* gy, float* gw, void* workspace, int B, int C, int O, int Df, int Hf, int Wf, void* stream) {
    return cv_stem_bwd(g, pre, consts, x, y, w, gx, gy, gw, static_cast<float*>(workspace), B, C, O, Df, Hf, Wf, ST(stream));
}
RAG_API int rag_conv3d_c1_fwd(const float* in, const float* w, float* out, int B, int C, int D, int H, int W, void* stream) {
    return conv3d_c1_fwd(in, w, out, B, C, D, H, W, ST(stream));
}
RAG_API size_t rag_conv3d_c1_bwd_workspace_bytes(int C) { return conv3d_c1_bwd_workspace_bytes(C); }
RAG_API int rag_conv3d_c1_bwd(const float* g, const float* in, const float* w, float* gin, float* gw, void* workspace,
                      int B, int C, int D, int H, int W, void* stream) {
    return conv3d_c1_bwd(g, in, w, gin, gw, static_cast<float*>(workspace), B, C, D, H, W, ST(stream));
}
RAG_API int rag_conv3d_cc_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                      int B, int C, int O, int D, int H, int W, void* stream) {
    return conv3d_cc_fwd(in, w, scale, shift, relu, out, B, C, O, D, H, W, ST(stream));
}
RAG_API size_t rag_conv3d_cc_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W) { return conv3d_cc_bwd_workspace_bytes(B, C, O, D, H, W); }
RAG_API int rag_conv3d_cc_bwd(const float* gz, const float* in, const float* w, float* gin, float* gw, void* workspace,
                      int B, int C, int O, int D, int H, int W, void* stream) {
    return conv3d_cc_bwd(gz, in, w, gin, gw, static_cast<float*>(workspace), B, C, O, D, H, W, ST(stream));
}
RAG_API int rag_conv3d_pw_fwd(const float* in, const float* w, const float* scale, const float* shift, int relu, float* out,
                      int B, int C, int O, int D, int H, int W, void* stream) {
    return conv3d_pw_fwd(in, w, scale, shift, relu, out, B, C, O, D, H, W, ST(stream));
}
RAG_API size_t rag_conv3d_pw_bwd_workspace_bytes(int B, int C, int O, int D, int H, int W) { return conv3d_pw_bwd_workspace_bytes(B, C, O, D, H, W); }
RAG_API int rag_conv3d_pw_bwd(const float* g, const float* z, const float* consts, const float* in, const float* w, float* gin, float* gw,
                      void* workspace, int B, int C, int O, int D, int H, int W, void* stream) {
    return conv3d_pw_bwd(g, z, consts, in, w, gin, gw, static_cast<float*>(workspace), B, C, O, D, H, W, ST(stream));
}
RAG_API int rag_bn3d_moments(const float* z, double* sums, double* rows_ws, int B, int O, int D, int H, int W, void* stream) {
    return bn3d_moments(z, sums, rows_ws, B, O, D, H, W, ST(stream));
}
RAG_API int rag_bn3d_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                      float* bn, int O, double n, double eps, double momentum, int batch, int update, void* stream) {
    return bn3d_finalize(sums, gamma, beta, running_mean, running_var, bn, O, n, eps, momentum, batch, update, ST(stream));
}
RAG_API int rag_bn3d_relu(float* z, const float* bn, int B, int O, int D, int H, int W, void* stream) {
    return bn3d_relu(z, bn, B, O, D, H, W, ST(stream));
}
RAG_API int rag_bn3d_bwd_sums(const float* g, const float* z, const float* bn, double* sums, double* rows_ws,
                      int B, int O, int D, int H, int W, void* stream) {
    return bn3d_bwd_sums(g, z, bn, sums, rows_ws, B, O, D, H, W, ST(stream));
}
RAG_API int rag_bn3d_bwd_consts(const double* sums, const float* bn, float* consts, float* gparam, int O, double n, int batch, void* stream) {
    return bn3d_bwd_consts(sums, bn, consts, gparam, O, n, batch, ST(stream));
}
RAG_API int rag_bn3d_bwd_gz(const float* g, const float* z, const float* consts, float* gz, int B, int O, int D, int H, int W, void* stream) {
    return bn3d_bwd_gz(g, z, consts, gz, B, O, D, H, W, ST(stream));
}
RAG_API int rag_trilinear_resize_fwd(const float* in, float* out, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners, void* stream) {
    return trilinear_resize_fwd(in, out, BC, Di, Hi, Wi, Do, Ho, Wo, align_corners, ST(stream));
}
RAG_API int rag_trilinear_resize_bwd(const float* gout, float* gin, int BC, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int align_corners, void* stream) {
    return trilinear_resize_bwd(gout, gin, BC, Di, Hi, Wi, Do, Ho, Wo, align_corners, ST(stream));
}
RAG_API int rag_bilinear_resize_fwd(const float* in, float* out, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners, void* stream) {
    return bilinear_resize_fwd(in, out, BC, Hi, Wi, Ho, Wo, align_corners, ST(stream));
}
RAG_API int rag_bilinear_resize_bwd(const float* gout, float* gin, int BC, int Hi, int Wi, int Ho, int Wo, int align_corners, void* stream) {
    return bilinear_resize_bwd(gout, gin, BC, Hi, Wi, Ho, Wo, align_corners, ST(stream));
}
RAG_API int rag_grid_sample_fwd(const float* in, const float* grid, float* out, int N, int C, int Hi, int Wi, int Ho, int Wo,
                        int padding_mode, int align_corners, void* stream) {
    return grid_sample_fwd(in, grid, out, N, C, Hi, Wi, Ho, Wo, padding_mode, align_corners, ST(stream));
}
RAG_API size_t rag_grid_sample_bwd_workspace_bytes(int N, int C, int Hi, int Wi, int Ho, int Wo) {
    return grid_sample_bwd_workspace_bytes(N, C, Hi, Wi, Ho, Wo);
}
RAG_API int rag_grid_sample_bwd(const float* gout, const float* in, const float* grid, float* gin, float* ggrid, void* workspace,
                        size_t workspace_bytes, int N, int C, int Hi, int Wi, int Ho, int Wo, int padding_mode, int align_corners,
                        void* stream) {
    return grid_sample_bwd(gout, in, grid, gin, ggrid, workspace, workspace_bytes, N, C, Hi, Wi, Ho, Wo, padding_mode, align_corners, ST(stream));
}
RAG_API int rag_normalize_pad(const uint8_t* img, float* out, int B, int H, int W, int top_pad, int right_pad, void* stream) {
    return normalize_pad(img, out, B, H, W, top_pad, right_pad, ST(stream));
}

}  // extern "C"
