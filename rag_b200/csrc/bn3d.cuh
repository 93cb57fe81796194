// The one expression of the BatchNorm3d + ReLU backward that every kernel forming the gradient at a convolution output uses
// (bn3d.cu's gz pass, conv3d_pw.cu's fused backward): the ReLU decision must be the forward's own fma(z, scale, shift) > 0,
// bit for bit, wherever it is re-evaluated.
#pragma once

namespace rag {

// gz = a (g' - m1 - zh m2) with g' = g [fma(z, sc, sh) > 0] and zh = (z - mu) rs; (a, m1, m2, sc, sh, mu, rs) = one row of the
// [O,7] consts of bn3d_bwd_consts
__device__ __forceinline__ float bn3d_gz(float g, float z, float a, float m1, float m2, float sc, float sh, float mu, float rs) {
    return a * ((__fmaf_rn(z, sc, sh) > 0.f ? g : 0.f) - m1 - ((z - mu) * rs) * m2);
}

}  // namespace rag
