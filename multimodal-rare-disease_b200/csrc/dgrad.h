// Data gradients through the frozen ResNet50 backbone (input saliency, Grad-CAM below layer4): the kernels of the
// backward that are not convolutions on the tcgen05 GEMM (those are plan_conv_dgrad, gemm_conv.h).  Everything is
// NHWC bf16 like the forward, except the stem's output, which is the caller's fp32 NCHW image gradient.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace mrd {

// Weights of a data-gradient convolution (plan_conv_dgrad's B operand) from a packed forward filter:
// w: [Cout][kk][Cin] bf16 (BatchNorm folded, the forward's pack) -> out: [Cin][ntaps][Cout] bf16 with
// out[ci][t][co] = w[co][src_tap[t]][ci].  kk in {1, 9}, ntaps <= 9.
struct TapList {
    int n;
    int tap[9];
};
int pack_dgrad_weights(const __nv_bfloat16* w, int Cout, int Cin, int kk, TapList src, __nv_bfloat16* out,
                       cudaStream_t s);

// gz = g * [y > 0] (backward of the ReLU that produced y), n elements, n % 8 == 0.
int relu_mask_bf16(const __nv_bfloat16* g, const __nv_bfloat16* y, long long n, __nv_bfloat16* gz, cudaStream_t s);

// Backward of AdaptiveAvgPool2d(1) followed by the block output's ReLU: gz[n,p,c] = d_pooled[n,c] / HW * [y[n,p,c] > 0].
// y: [N,HW,C] bf16, d_pooled: [N,C] fp32, C % 8 == 0.
int avgpool_bwd_mask_bf16(const float* d_pooled, int N, int HW, int C, const __nv_bfloat16* y, __nv_bfloat16* gz,
                          cudaStream_t s);

// Backward of MaxPool2d(3, 2, 1) (TV:models/resnet.py:200,271) fused with the backward of the ReLU in front of it.
// y: [N,H,W,C] bf16 = the pooled tensor (post-ReLU), g: [N,H/2,W/2,C] bf16 = d(loss)/d(pool output).
// dx[n,h,w,c] = [y > 0] * sum of g over the windows whose maximum is (h, w) - the first maximum of the window in
// row-major order, as PyTorch's max_pool2d_with_indices picks it.  Every element is gathered by one thread (no atomics:
// the result does not depend on the schedule).  H, W even, C % 8 == 0.
int maxpool3x3s2_bwd_relu(const __nv_bfloat16* g, const __nv_bfloat16* y, int N, int H, int W, int C,
                          __nv_bfloat16* dx, cudaStream_t s);

// Stem filter with BatchNorm folded, laid out for stem_dgrad_nchw: w [64,3,7,7] fp32 -> out [7][7][64][3] fp32,
// out[kh][kw][co][c] = w[co][c][kh][kw] * gamma[co] / sqrt(var[co] + eps).
int pack_stem_dgrad(const float* w, const float* gamma, const float* var, float eps, float* out, cudaStream_t s);

// Data gradient of the 7x7 / stride-2 / pad-3 stem convolution (3 -> 64 channels), written as the caller's image
// gradient: d: [N,H/2,W/2,64] bf16 (d(loss)/d(conv output)), wf: pack_stem_dgrad, out: [N,3,H,W] fp32.  CUDA cores:
// 0.24 GFLOP per 224 x 224 image, 3 % of the backbone's backward.  H, W even.
int stem_dgrad_nchw(const __nv_bfloat16* d, const float* wf, int N, int H, int W, float* out, cudaStream_t s);

}  // namespace mrd
